"""Encoder hot spot on the B200 (SURVEY.md 8(f) rank 4): the gating neural adaptive bias of an attention-free block.

`DistAngleFusion` mirrors `rrnco/models/nn/attn_freenet.py:201-289` (same constructor, same parameter names, so the
reference module's state_dict loads unchanged); its forward is ONE kernel (`rrnco_nab_gating`) that never materialises the
[B, N, N, E] embeddings upstream builds twice per block.  `patch_encoder` swaps it into an upstream `RRNetEncoder`
(`encoder.net.layers[i].{row,col}_encoding_block.angle_distance_fusion`) for the inference path (test.py / validation), and
with `trainable=True` for training too: the backward of the two-way gate is one pass over the node pairs as well
(`rrnco_train_nab_backward`, csrc_train/encoder_train.cu), so autograd keeps [B, N, N] tensors, not seven [B, N, N, E] ones.
The duration-channel variant (rcvrptw: Linear(3E, E) -> SiLU -> Linear(E, 3) gate, softmax with a temperature) does not
collapse to scalar functions (its gate is not linear in the embeddings): what remains after collapsing the linear layers is a
[pairs x 3E] x [3E x E] contraction, which runs on tcgen05 (`rrnco_nab_dur_gating`, csrc/encoder_dur_kernel.cu).  With
`train_duration_gate=True` it trains too: its backward (`rrnco_train_nab_dur_backward`, csrc_train/encoder_dur_train.cu) is
six E x E contractions over the pairs on tcgen05 plus small sums, so autograd keeps [B, N, N] tensors, not twelve
[B, N, N, E] ones.
No CPU fallback: a host tensor or a missing library raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import nn

from . import _lib, train_ops
from ._lib import call, ptr, stream_ptr


def _nab_params(m: "DistAngleFusion"):
    """The 12 tensors of a two-way-gate module in the order of rrnco_train_nab_backward's `params` / `grads`."""
    return [m.dist_emb[0].weight, m.dist_emb[0].bias, m.dist_emb[2].weight, m.dist_emb[2].bias,
            m.angle_emb[0].weight, m.angle_emb[0].bias, m.angle_emb[2].weight, m.angle_emb[2].bias,
            m.gate[0].weight, m.gate[0].bias, m.out_lin.weight, m.out_lin.bias]


def _dur_params(m: "DistAngleFusion"):
    """The 19 tensors of a duration-gate module in the pointer order of rrnco_nab_dur_pack (= rrnco_train_nab_dur_backward's
    `params` / `grads`)."""
    return [*(q for seq in (m.dist_emb, m.angle_emb, m.dur_emb) for q in (seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias)),
            m.gate[0].weight, m.gate[0].bias, m.gate[2].weight, m.gate[2].bias, m.gate_temperature,
            m.out_lin.weight, m.out_lin.bias]


_train_checked = False
_dur_train_checked = False


def _train_lib():
    """librrnco_b200_train.so, once checked to read `packed` in the layout the rollout library writes it."""
    global _train_checked
    h = train_ops.lib()
    if not _train_checked:
        if h.rrnco_train_nab_packed_floats() != _lib.lib().rrnco_nab_packed_floats():
            raise RuntimeError("librrnco_b200_train.so and librrnco_b200.so disagree on the layout of the packed "
                               "DistAngleFusion tables: rebuild both (python rrnco_b200/build.py --force)")
        _train_checked = True
    return h


def _dur_train_lib():
    """librrnco_b200_train.so, once checked to read the duration gate's `packed` in the layout the rollout library writes."""
    global _dur_train_checked
    h = train_ops.lib()
    if not _dur_train_checked:
        if h.rrnco_train_nab_dur_packed_bytes() != _lib.lib().rrnco_nab_dur_packed_bytes():
            raise RuntimeError("librrnco_b200_train.so and librrnco_b200.so disagree on the layout of the packed "
                               "duration-gate tables: rebuild both (python rrnco_b200/build.py --force)")
        _dur_train_checked = True
    return h


def nab_dur_gating_backward(coords: torch.Tensor, cost: torch.Tensor, dur: torch.Tensor, transposed: int,
                            packed: torch.Tensor, flat_params: torch.Tensor, scale: float,
                            grad_out: torch.Tensor) -> torch.Tensor:
    """Parameter gradients of the duration gate (rrnco_train_nab_dur_backward) as one flat fp32 tensor in the layout of
    `_dur_params`: `coords`, `cost` / `dur` (the contiguous bases, read transposed when `transposed`), `packed` and `scale`
    as the forward call got them, `flat_params` the 19 parameters concatenated, `grad_out` [B, N, N].  An fp16 operand
    overflow or a non-finite value raises."""
    h, dev = _dur_train_lib(), cost.device
    B, N, _ = cost.shape
    nbytes = h.rrnco_train_nab_dur_workspace_bytes(B, N)
    train_ops._check(min(nbytes, 0), "rrnco_train_nab_dur_workspace_bytes")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    grads = torch.empty(h.rrnco_train_nab_dur_grad_floats(), dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    grad_out = grad_out.float().contiguous()
    train_ops._check(h.rrnco_train_nab_dur_backward(B, N, ptr(coords), ptr(cost), ptr(dur), int(transposed), ptr(packed),
                                                    ptr(flat_params), float(scale), ptr(grad_out), ptr(ws), ptr(grads),
                                                    ptr(status), stream_ptr(dev)),
                     "rrnco_train_nab_dur_backward")
    if int(status.item()):
        raise AssertionError("DistAngleFusion backward: an fp16 operand overflowed (pair scalar >= 4094 or a gradient far "
                             "outside the range of the others) or a value is not finite")
    return grads


def nab_gating_backward(coords: torch.Tensor, cost: torch.Tensor, transposed: int, packed: torch.Tensor,
                        flat_params: torch.Tensor, scale: float, grad_out: torch.Tensor) -> torch.Tensor:
    """Parameter gradients of the two-way gate (rrnco_train_nab_backward) as one flat fp32 tensor in the layout of
    `_nab_params`: `coords`, `cost` (the contiguous base, read transposed when `transposed`), `packed` and `scale` as the
    forward call got them, `flat_params` the 12 parameters concatenated, `grad_out` [B, N, N]."""
    h, dev = _train_lib(), cost.device
    B, N, _ = cost.shape
    nbytes = h.rrnco_train_nab_workspace_bytes(B, N)
    train_ops._check(min(nbytes, 0), "rrnco_train_nab_workspace_bytes")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    grads = torch.empty(h.rrnco_train_nab_grad_floats(), dtype=torch.float32, device=dev)
    grad_out = grad_out.float().contiguous()
    train_ops._check(h.rrnco_train_nab_backward(B, N, ptr(coords), ptr(cost), int(transposed), ptr(packed), ptr(flat_params),
                                                float(scale), ptr(grad_out), ptr(ws), ptr(grads), stream_ptr(dev)),
                     "rrnco_train_nab_backward")
    return grads


class _NabGating(torch.autograd.Function):
    """out = DistAngleFusion.forward (two-way gate) through rrnco_nab_gating; backward = rrnco_train_nab_backward.  The
    context keeps the `packed` buffer the forward used (a parameter update makes the module pack a NEW buffer) and a snapshot
    of the parameters; no gradients flow to coords / cost."""

    @staticmethod
    def forward(ctx, coords, cost, transposed, scale, packed, *params):
        B, N, _ = cost.shape
        out = torch.empty((B, N, N), dtype=torch.float32, device=cost.device)
        call("rrnco_nab_gating", B, N, ptr(coords), ptr(cost), transposed, ptr(packed), float(scale), 0, ptr(out),
             stream_ptr(cost.device))
        flat = torch.cat([p.detach().float().reshape(-1) for p in params])
        ctx.save_for_backward(coords, cost, packed, flat)
        ctx.transposed, ctx.scale = transposed, float(scale)
        ctx.metas = [(p.shape, p.dtype) for p in params]
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        coords, cost, packed, flat = ctx.saved_tensors
        with torch.cuda.device(cost.device):
            grads = nab_gating_backward(coords, cost, ctx.transposed, packed, flat, ctx.scale, grad_out)
        out, off = [], 0
        for shape, dtype in ctx.metas:
            n = shape.numel()
            out.append(grads[off:off + n].view(shape).to(dtype))
            off += n
        return (None, None, None, None, None, *out)


class _NabDurGating(torch.autograd.Function):
    """out = DistAngleFusion.forward (duration gate) through rrnco_nab_dur_gating, with its status check; backward =
    rrnco_train_nab_dur_backward.  The context keeps the `packed` buffer the forward used and a snapshot of the parameters;
    no gradients flow to coords / cost / duration."""

    @staticmethod
    def forward(ctx, coords, cost, dur, transposed, scale, packed, check, *params):
        B, N, _ = cost.shape
        out = torch.empty((B, N, N), dtype=torch.float32, device=cost.device)
        status = torch.zeros(1, dtype=torch.int32, device=cost.device)
        call("rrnco_nab_dur_gating", B, N, ptr(coords), ptr(cost), ptr(dur), transposed, ptr(packed), float(scale), ptr(out),
             ptr(status), stream_ptr(cost.device))
        if check and int(status.item()):
            raise AssertionError("DistAngleFusion: hidden activations outside the fp16 operand range (>= 4094) "
                                 "or a cost / duration / coordinate that is not finite")
        flat = torch.cat([p.detach().float().reshape(-1) for p in params])
        ctx.save_for_backward(coords, cost, dur, packed, flat)
        ctx.transposed, ctx.scale = transposed, float(scale)
        ctx.metas = [(p.shape, p.dtype) for p in params]
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        coords, cost, dur, packed, flat = ctx.saved_tensors
        with torch.cuda.device(cost.device):
            grads = nab_dur_gating_backward(coords, cost, dur, ctx.transposed, packed, flat, ctx.scale, grad_out)
        out, off = [], 0
        for shape, dtype in ctx.metas:
            n = shape.numel()
            out.append(grads[off:off + n].view(shape).to(dtype))
            off += n
        return (None, None, None, None, None, None, None, *out)


class DistAngleFusion(nn.Module):
    def __init__(self, embed_dim: int = 128, use_duration_matrix: bool = False, trainable: bool = False,
                 train_duration_gate: bool = False):
        """`trainable=True`: under grad (with parameters that require it) the forward records an autograd node whose
        backward is a CUDA kernel (rrnco_train_nab_backward); every other call is the inference kernel.  The duration gate
        (`use_duration_matrix=True`) trains only with `train_duration_gate=True` as well (rrnco_train_nab_dur_backward)."""
        super().__init__()
        if embed_dim != 128:
            raise NotImplementedError("the kernels are built for embed_dim = 128 (experiment/rrnet.yaml)")
        if trainable and use_duration_matrix and not train_duration_gate:
            raise NotImplementedError("trainable=True: the backward kernel covers the two-way gate (ATSP / RCVRP); the "
                                      "rcvrptw duration gate trains with train_duration_gate=True")
        self.trainable = bool(trainable)
        self.use_duration_matrix = bool(use_duration_matrix)
        self.embed_dim = embed_dim // 2 if use_duration_matrix else embed_dim  # (upstream's attribute, attn_freenet.py:210-214)
        self.dist_emb = nn.Sequential(nn.Linear(1, embed_dim), nn.ReLU(), nn.Linear(embed_dim, embed_dim))
        self.angle_emb = nn.Sequential(nn.Linear(1, embed_dim), nn.ReLU(), nn.Linear(embed_dim, embed_dim))
        if use_duration_matrix:  # attn_freenet.py:226-238
            self.dur_emb = nn.Sequential(nn.Linear(1, embed_dim), nn.ReLU(), nn.Linear(embed_dim, embed_dim))
            self.gate = nn.Sequential(nn.Linear(3 * embed_dim, embed_dim), nn.SiLU(), nn.Linear(embed_dim, 3))
            self.gate_temperature = nn.Parameter(torch.tensor(5.0))
        else:
            self.gate = nn.Sequential(nn.Linear(embed_dim * 2, 1), nn.Sigmoid())
        self.out_lin = nn.Linear(embed_dim, 1)
        self._packed = None
        self._packed_key = None
        self._keep = None
        self.check_overflow = True  # read the kernel's status word back after each duration-gate call (one host sync)

    def _packed_duration(self) -> torch.Tensor:
        ps = [*(m for seq in (self.dist_emb, self.angle_emb, self.dur_emb) for m in (seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias)),
              self.gate[0].weight, self.gate[0].bias, self.gate[2].weight, self.gate[2].bias, self.gate_temperature,
              self.out_lin.weight, self.out_lin.bias]
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if self._packed is None or self._packed_key != key:
            dev = ps[0].device
            cont = [p.detach().float().contiguous().reshape(-1) for p in ps]
            ptrs = torch.tensor([c.data_ptr() for c in cont], dtype=torch.int64, device=dev)
            packed = torch.empty(_lib.lib().rrnco_nab_dur_packed_bytes(), dtype=torch.uint8, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            call("rrnco_nab_dur_pack", ptr(ptrs), ptr(packed), ptr(status), stream_ptr(dev))
            if int(status.item()):
                raise AssertionError("DistAngleFusion: collapsed gate weights outside the fp16 operand range (|w| >= 255)")
            self._packed, self._packed_key, self._keep = packed, key, cont
        return self._packed

    def packed_parameters(self) -> torch.Tensor:
        """The module collapsed into four E-vectors + constants (rrnco_nab_pack); cached until a parameter changes."""
        ps = _nab_params(self)
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if self._packed is None or self._packed_key != key:
            dev = ps[0].device
            packed = torch.empty(_lib.lib().rrnco_nab_packed_floats(), dtype=torch.float32, device=dev)
            cont = [p.detach().float().contiguous() for p in ps]
            call("rrnco_nab_pack", *[ptr(p) for p in cont], ptr(packed), stream_ptr(dev))
            self._packed, self._packed_key = packed, key
        return self._packed

    def forward(self, coords: torch.Tensor, cost_mat: torch.Tensor, duration_mat=None, scale: float = 1.0,
                variant: int = 0) -> torch.Tensor:
        """adapt_bias [B, N, N] (times `scale`, e.g. the block's alpha).  `cost_mat` may be the transposed VIEW the
        col-encoding block passes (attn_freenet.py:480-486): it is read through its base, never copied.
        `variant` 0 = piecewise-linear segment tables (default), 1 = brute-force sum over the hidden units (cross-check)."""
        record = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if record and not self.trainable:
            raise NotImplementedError("forward-only kernel: call under torch.no_grad() / inference_mode (test.py path)")
        if record and variant != 0:
            raise NotImplementedError("trainable DistAngleFusion: the backward kernel follows the segment tables (variant 0)")
        if record and (coords.requires_grad or cost_mat.requires_grad):
            raise NotImplementedError("trainable DistAngleFusion: no gradients with respect to coords / cost_mat")
        if (duration_mat is not None) != self.use_duration_matrix:
            raise ValueError("duration_mat must be given exactly when the module was built with use_duration_matrix=True")
        B, N, _ = cost_mat.shape
        coords = coords.float().contiguous()
        transposed = 0
        if not cost_mat.is_contiguous() and cost_mat.transpose(1, 2).is_contiguous():
            cost_mat, transposed = cost_mat.transpose(1, 2), 1
        cost_mat = cost_mat.float().contiguous()
        if record and not self.use_duration_matrix:
            return _NabGating.apply(coords, cost_mat, transposed, float(scale), self.packed_parameters(), *_nab_params(self))
        out = torch.empty((B, N, N), dtype=torch.float32, device=cost_mat.device)
        if self.use_duration_matrix:  # three-way gate: tcgen05 kernel (encoder_dur_kernel.cu)
            dur = duration_mat
            if transposed:  # the col-encoding block transposes both matrices (attn_freenet.py:476-486)
                dur = dur.transpose(1, 2)
            dur = dur.float().contiguous()
            if record:
                if duration_mat.requires_grad:
                    raise NotImplementedError("trainable DistAngleFusion: no gradients with respect to duration_mat")
                return _NabDurGating.apply(coords, cost_mat, dur, transposed, float(scale), self._packed_duration(),
                                           self.check_overflow, *_dur_params(self))
            status = torch.zeros(1, dtype=torch.int32, device=out.device)
            call("rrnco_nab_dur_gating", B, N, ptr(coords), ptr(cost_mat), ptr(dur), transposed, ptr(self._packed_duration()),
                 float(scale), ptr(out), ptr(status), stream_ptr(out.device))
            if self.check_overflow and int(status.item()):
                raise AssertionError("DistAngleFusion: hidden activations outside the fp16 operand range (>= 4094) "
                                     "or a cost / duration / coordinate that is not finite")
            return out
        call("rrnco_nab_gating", B, N, ptr(coords), ptr(cost_mat), transposed, ptr(self.packed_parameters()), float(scale),
             int(variant), ptr(out), stream_ptr(cost_mat.device))
        return out


def aft_nab(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, coords, cost_mat: torch.Tensor,
            fusion: Optional[DistAngleFusion], scale: float = 1.0) -> torch.Tensor:
    """The O(N^2) part of an attention-free block in one kernel (`rrnco_aft_nab`): the neural adaptive bias
    (`fusion`, times `scale` = the block's alpha), its row softmax and exp, exp(softmax over the tokens of k), the two
    [N,N] x [N,E] products and the sigmoid(q) gate -- `AFTFull.forward` (attn_freenet.py:309-327) without its Linear layers:
    q / k / v are to_q(x) / to_k(y) / to_v(y) and the caller applies `project`.  N <= 128; nothing of size [B,N,N] is written.
    `fusion=None`: `cost_mat` IS the adapt_bias [B,N,N] (any gate variant, e.g. the duration gate's output), `coords` unused."""
    B, N, E = q.shape
    if N > 128:
        raise NotImplementedError("rrnco_aft_nab holds the instance's key tiles in shared memory: N <= 128 "
                                  "(use DistAngleFusion + torch for larger instances)")
    if torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad):
        raise NotImplementedError("forward-only kernel: call under torch.no_grad() / inference_mode (test.py path)")
    q, k, v = q.float().contiguous(), k.float().contiguous(), v.float().contiguous()
    coords = None if fusion is None else coords.float().contiguous()
    transposed = 0
    if not cost_mat.is_contiguous() and cost_mat.transpose(1, 2).is_contiguous():
        cost_mat, transposed = cost_mat.transpose(1, 2), 1
    cost_mat = cost_mat.float().contiguous()
    out = torch.empty_like(q)
    call("rrnco_aft_nab", B, N, ptr(q), ptr(k), ptr(v), ptr(coords), ptr(cost_mat), transposed,
         ptr(None if fusion is None else fusion.packed_parameters()), float(scale), ptr(out), stream_ptr(q.device))
    return out


def _fused_block_forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None):
    """AttnFree_Block.forward (attn_freenet.py:417-442) with the bias + AFT-full part as one kernel; everything else
    (norms, Linear layers, feed-forward) is the block's own modules, unchanged."""
    row_emb = self.norm1(row_emb)
    col_emb = self.norm2(col_emb)
    aft = self.attn_free
    if duration_mat is not None:  # rcvrptw: bias from the tcgen05 gate kernel, then the fused AFT-full over it
        bias = self.neural_adaptive_bias(coords, cost_mat, duration_mat, scale=float(self.alpha))
        y = aft_nab(aft.to_q(row_emb), aft.to_k(col_emb), aft.to_v(col_emb), None, bias, None, 1.0)
    else:
        y = aft_nab(aft.to_q(row_emb), aft.to_k(col_emb), aft.to_v(col_emb), coords, cost_mat, self.angle_distance_fusion,
                    float(self.alpha))
    out_concat = aft.project(y)
    multi_head_out = self.norm3(self.multi_head_combine(out_concat))
    return self.feed_forward(multi_head_out, row_emb)


def patch_encoder(encoder: nn.Module, fuse_aft: bool = True, trainable: bool = False, train_duration_gate: bool = False) -> int:
    """Replaces every gating `DistAngleFusion` without duration channel inside an upstream encoder (attribute
    `angle_distance_fusion` of the attention-free blocks, attn_freenet.py:386-389) by the kernel-backed module with the
    same parameters, and (fuse_aft, instances of <= 128 nodes) routes the block's bias -> AFT-full chain through the fused
    kernel.  Inference path only, unless `trainable`: then the swapped modules are `DistAngleFusion(trainable=True)` that
    hold upstream's own parameter tensors (an optimizer built before the patch keeps training them), the rcvrptw
    duration-gate modules stay upstream's, and the fused block runs under torch.no_grad() only (under grad the block is
    upstream's forward around the trainable module).  With `train_duration_gate` as well, the rcvrptw modules are swapped
    too, for `DistAngleFusion(use_duration_matrix=True, trainable=True, train_duration_gate=True)` holding upstream's 19
    parameter tensors (gate_temperature included).  Returns the number of blocks patched."""
    import types
    n = 0
    for block in encoder.modules():
        if trainable and not train_duration_gate and hasattr(getattr(block, "neural_adaptive_bias", None), "dur_emb"):
            continue
        # rcvrptw blocks: attribute `neural_adaptive_bias` holding a DistAngleFusion with the duration channel (:380-384)
        refd = getattr(block, "neural_adaptive_bias", None)
        if refd is not None and not isinstance(refd, DistAngleFusion) and hasattr(refd, "dur_emb") and hasattr(refd, "gate_temperature"):
            mine = DistAngleFusion(128, use_duration_matrix=True, trainable=trainable,
                                   train_duration_gate=trainable).to(next(refd.parameters()).device)
            mine.load_state_dict(refd.state_dict(), strict=True)
            if trainable:  # upstream's own tensors: an optimizer built before the patch keeps training them
                mine.dist_emb, mine.angle_emb, mine.dur_emb, mine.gate, mine.out_lin = (
                    refd.dist_emb, refd.angle_emb, refd.dur_emb, refd.gate, refd.out_lin)
                mine.gate_temperature = refd.gate_temperature
            block.neural_adaptive_bias = mine
            if fuse_aft and all(hasattr(block, a) for a in ("attn_free", "norm1", "norm2", "norm3", "multi_head_combine",
                                                            "feed_forward", "alpha")):
                unfused_d = block.forward

                def forward_d(self, row_emb, col_emb, cost_mat, coords, duration_mat=None, _unfused=unfused_d):
                    if cost_mat.shape[-1] > 128 or duration_mat is None or torch.is_grad_enabled():
                        return _unfused(row_emb, col_emb, cost_mat, coords, duration_mat)
                    return _fused_block_forward(self, row_emb, col_emb, cost_mat, coords, duration_mat)
                block.forward = types.MethodType(forward_d, block)
            n += 1
            continue
        ref = getattr(block, "angle_distance_fusion", None)
        if ref is None or isinstance(ref, DistAngleFusion) or hasattr(ref, "dur_emb"):
            continue
        mine = DistAngleFusion(ref.embed_dim, trainable=trainable).to(next(ref.parameters()).device)
        mine.load_state_dict(ref.state_dict(), strict=True)
        if trainable:
            mine.dist_emb, mine.angle_emb, mine.gate, mine.out_lin = ref.dist_emb, ref.angle_emb, ref.gate, ref.out_lin
        block.angle_distance_fusion = mine
        if fuse_aft and all(hasattr(block, a) for a in ("attn_free", "norm1", "norm2", "norm3", "multi_head_combine",
                                                        "feed_forward", "alpha")):
            unfused = block.forward

            def forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None, _unfused=unfused):
                if cost_mat.shape[-1] > 128 or duration_mat is not None or torch.is_grad_enabled():
                    return _unfused(row_emb, col_emb, cost_mat, coords, duration_mat)
                return _fused_block_forward(self, row_emb, col_emb, cost_mat, coords, duration_mat)
            block.forward = types.MethodType(forward, block)
        n += 1
    return n
