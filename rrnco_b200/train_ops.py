"""ctypes binding of librrnco_b200_train.so (include/rrnco_b200_train.h) and the autograd Functions built on it: the heavy
parts of the training hand-off (`training.batched_logprobs`) as hand-written sm_100a kernels, forward AND backward.

    fused_ffn(x, w1, b1, w2, b2)             residual FFN of the pointer (decoder.py:272-277, 296) on tcgen05, fp32-faithful
    fused_attention(q, k, v, mask)           masked 8-head attention + residual (decoder.py:281-293), N <= 1024
    pointer_scores(g, lk) / pointer_logprob  pointer scores g . Lk^T on tcgen05 (decoder.py:298-301), N <= 1024
    fused_logits_tail(z, decoder, ...)       edge bias / log(exp + 1e-6) / tanh clip / mask / log-softmax / gather
                                             (decoder.py:183-198, decoding.py:311-399)

No CPU fallback: a missing library or a CPU tensor raises.  Torch is used for device memory, streams and the autograd graph.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librrnco_b200_train.so")
MAX_NODES_ATTENTION = 102   # K, V, dK, dV tiles of one instance in shared memory (rrnco_train_attention_bwd); above: key-tiled kernels
MAX_NODES_POINTER = 128     # one 128 x 128 weight tile per instance (rrnco_train_inst_*); above: ceil(N / 128) key tiles
MAX_NODES_REPLAY = 1024     # largest instance of the key-tiled kernels (rrnco_train_attention_tiled_*, rrnco_train_inst_tiled_*)
DEV_NAN_LOGITS = 1

_f = C.c_void_p
_SIGNATURES = {
    "rrnco_train_ffn_packed_bytes": (C.c_int64, []),
    "rrnco_train_ffn_pack": (C.c_int, [_f, _f, _f, _f, _f]),
    "rrnco_train_ffn": (C.c_int, [C.c_int32, C.c_int64, _f, _f, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_xty": (C.c_int, [C.c_int64, _f, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_attention_fwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, C.c_int32, _f, _f, _f]),
    "rrnco_train_attention_bwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, _f, C.c_int32, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_attention_tiled_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int32]),
    "rrnco_train_attention_tiled_fwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, C.c_int32, _f, _f, _f]),
    "rrnco_train_attention_tiled_bwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, _f, C.c_int32, _f, _f, _f, _f, _f,
                                                  _f, _f]),
    "rrnco_train_context_query_fwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, _f, C.c_int32, _f, _f, _f]),
    "rrnco_train_context_query_bwd": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, C.c_int32, _f, _f, _f, _f]),
    "rrnco_train_logits_tail": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f, C.c_float, C.c_float,
                                          C.c_float, _f, _f, _f, _f]),
    "rrnco_train_inst_packed_bytes": (C.c_int64, [C.c_int64]),
    "rrnco_train_inst_pack": (C.c_int, [C.c_int64, C.c_int32, _f, C.c_int32, _f, _f, _f]),
    "rrnco_train_inst_gemm": (C.c_int, [C.c_int64, C.c_int64, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_inst_xty": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_inst_tiled_packed_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "rrnco_train_inst_tiled_pack": (C.c_int, [C.c_int64, C.c_int32, _f, C.c_int32, _f, _f, _f]),
    "rrnco_train_inst_tiled_gemm": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_int32, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_inst_tiled_xty": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_train_nab_packed_floats": (C.c_int64, []),
    "rrnco_train_nab_grad_floats": (C.c_int64, []),
    "rrnco_train_nab_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "rrnco_train_nab_backward": (C.c_int, [C.c_int64, C.c_int32, _f, _f, C.c_int32, _f, _f, C.c_float, _f, _f, _f, _f]),
    "rrnco_train_nab_dur_packed_bytes": (C.c_int64, []),
    "rrnco_train_nab_dur_grad_floats": (C.c_int64, []),
    "rrnco_train_nab_dur_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "rrnco_train_nab_dur_backward": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, C.c_int32, _f, _f, C.c_float, _f, _f, _f, _f,
                                               _f]),
}
_lib = None
_status: dict = {}


def exported_symbols():
    return list(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python rrnco_b200/build.py` (there is no CPU fallback)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


def available() -> bool:
    return os.path.exists(LIB_PATH)


def _p(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("rrnco_b200.train_ops: CUDA tensors only (no CPU fallback)")
    return C.c_void_p(t.data_ptr())


def _on_device(fn):
    """Kernel launches go to the CURRENT device: run the wrapped forward / backward on the device of its first tensor argument
    (a process may hold tensors on several GPUs)."""
    import functools

    @functools.wraps(fn)
    def wrapped(ctx, *args):
        for a in args:
            if isinstance(a, torch.Tensor) and a.is_cuda:
                with torch.cuda.device(a.device):
                    return fn(ctx, *args)
        return fn(ctx, *args)
    return wrapped


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed with code {rc}")


def status_word(dev) -> torch.Tensor:
    """Sticky device word of this device: RRNCO_DEV_NAN_LOGITS when an fp16 operand overflowed in any call so far."""
    dev = torch.device(dev)
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _status:
        _status[key] = torch.zeros(1, dtype=torch.int32, device=dev)
    return _status[key]


def check_status(dev) -> None:
    """One device -> host read: raises if a kernel flagged an fp16 operand overflow since the last check."""
    w = status_word(dev)
    v = int(w.item())
    if v:
        w.zero_()
        raise FloatingPointError(f"rrnco_b200.train_ops: fp16 hi|lo operand overflow (status {v}): result not to be trusted")


def pow2_scale(t: torch.Tensor, bound_factor=None, target: float = 512.0) -> torch.Tensor:
    """Device scalar 2^k with max|t| * bound_factor * 2^k in (target / 2, target]: the pre-split scale of a gradient operand."""
    lo, hi = torch.aminmax(t.detach())          # one pass, nothing materialised (|t| would be a full copy)
    amax = torch.maximum(-lo, hi).float()
    if bound_factor is not None:
        amax = amax * bound_factor
    amax = amax.clamp(1e-30, 1e30)
    return torch.exp2(torch.floor(torch.log2(target / amax))).reshape(1).contiguous()


def _pack(wa, wb, dev):
    h = lib()
    packed = torch.empty(h.rrnco_train_ffn_packed_bytes(), dtype=torch.uint8, device=dev)
    _check(h.rrnco_train_ffn_pack(_p(wa), _p(wb), _p(packed), _p(status_word(dev)), _stream(dev)), "rrnco_train_ffn_pack")
    return packed


SAVE_HIDDEN = True   # keep the [rows, 512] hidden activations of the forward call for dW2 (2 KB per row) instead of recomputing them


class _FusedFFN(torch.autograd.Function):
    @staticmethod
    @_on_device
    def forward(ctx, x, w1, b1, w2, b2):
        h, dev = lib(), x.device
        x = x.detach().contiguous().float()
        w1, b1, w2, b2 = (t.detach().contiguous().float() for t in (w1, b1, w2, b2))
        rows = x.shape[0]
        mask = torch.empty(rows, 16, dtype=torch.int32, device=dev)
        y = torch.empty_like(x)
        keep = SAVE_HIDDEN and any(ctx.needs_input_grad)
        hidden = torch.empty((rows + 127) // 128 * 128 * 512, dtype=torch.float32, device=dev) if keep else None   # tile-blocked
        packed = _pack(w1, w2, dev)
        _check(h.rrnco_train_ffn(0, rows, _p(x), _p(packed), _p(b1), _p(b2), None, _p(mask), _p(hidden), _p(y),
                                 _p(status_word(dev)), _stream(dev)), "rrnco_train_ffn")
        ctx.save_for_backward(x, mask, w1, b1, w2, b2, hidden)
        return y

    @staticmethod
    @_on_device
    def backward(ctx, dy):
        x, mask, w1, b1, w2, b2, hidden = ctx.saved_tensors
        h, dev, st = lib(), x.device, status_word(x.device)
        rows = x.shape[0]
        dy = dy.contiguous().float()
        lo, hi = torch.aminmax(dy)
        amax = torch.maximum(-lo, hi)
        s_dy = pow2_scale(amax)
        # |dhidden_j| <= max|dy| * sum_e |W2[e, j]|: a rigorous bound without a pass over the [rows, 512] tensor
        s_dh = pow2_scale(amax, bound_factor=w2.abs().sum(0).amax().clamp_min(1.0))
        if hidden is None:
            hidden = torch.empty((rows + 127) // 128 * 128 * 512, dtype=torch.float32, device=dev)
            packed = _pack(w1, w2, dev)
            _check(h.rrnco_train_ffn(0, rows, _p(x), _p(packed), _p(b1), _p(b2), None, None, _p(hidden), None, _p(st),
                                     _stream(dev)), "rrnco_train_ffn (recompute)")
        dhid = torch.empty((rows + 127) // 128 * 128 * 512, dtype=torch.float32, device=dev)   # tile-blocked, as hidden
        dx = torch.empty_like(x)
        packed_t = _pack(w2.t().contiguous(), w1.t().contiguous(), dev)
        _check(h.rrnco_train_ffn(1, rows, _p(dy), _p(packed_t), None, None, _p(s_dy), _p(mask), _p(dhid), _p(dx), _p(st),
                                 _stream(dev)), "rrnco_train_ffn (backward)")
        dw1 = torch.zeros(512, 128, dtype=torch.float32, device=dev)
        db1 = torch.zeros(512, dtype=torch.float32, device=dev)
        dw2t = torch.zeros(512, 128, dtype=torch.float32, device=dev)
        db2 = torch.zeros(128, dtype=torch.float32, device=dev)
        _check(h.rrnco_train_xty(rows, _p(dhid), 1, _p(x), _p(s_dh), None, _p(dw1), _p(db1), None, _p(st), _stream(dev)),
               "rrnco_train_xty (dW1)")
        _check(h.rrnco_train_xty(rows, _p(hidden), 1, _p(dy), None, _p(s_dy), _p(dw2t), None, _p(db2), _p(st), _stream(dev)),
               "rrnco_train_xty (dW2)")
        return dx, dw1, db1, dw2t.t(), db2


def fused_ffn(x, w1, b1, w2, b2):
    """y = relu(x w1^T + b1) w2^T + b2 + x for x [..., 128]; forward, data and weight gradients on tcgen05 (fp32-faithful)."""
    return _FusedFFN.apply(x.reshape(-1, 128), w1, b1, w2, b2).view(x.shape)


class _FusedAttention(torch.autograd.Function):
    @staticmethod
    @_on_device
    def forward(ctx, q, k, v, mask, add_residual):
        h, dev = lib(), q.device
        q, k, v = (t.detach().contiguous().float() for t in (q, k, v))
        m8 = mask.contiguous().view(torch.uint8)
        n_inst, L, _ = q.shape
        N = k.shape[1]
        out = torch.empty_like(q)
        lse = torch.empty(n_inst, L, 8, dtype=torch.float32, device=dev)
        fwd = h.rrnco_train_attention_fwd if N <= MAX_NODES_ATTENTION else h.rrnco_train_attention_tiled_fwd
        _check(fwd(n_inst, L, N, _p(q), _p(k), _p(v), _p(m8), int(add_residual), _p(out), _p(lse), _stream(dev)),
               "rrnco_train_attention_fwd" if N <= MAX_NODES_ATTENTION else "rrnco_train_attention_tiled_fwd")
        ctx.save_for_backward(q, k, v, m8, out, lse)
        ctx.add_residual = int(add_residual)
        return out

    @staticmethod
    @_on_device
    def backward(ctx, d_out):
        q, k, v, m8, out, lse = ctx.saved_tensors
        h, dev = lib(), q.device
        n_inst, L, _ = q.shape
        N = k.shape[1]
        d_out = d_out.contiguous().float()
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        if N <= MAX_NODES_ATTENTION:
            _check(h.rrnco_train_attention_bwd(n_inst, L, N, _p(q), _p(k), _p(v), _p(m8), _p(out), ctx.add_residual, _p(lse),
                                               _p(d_out), _p(dq), _p(dk), _p(dv), _stream(dev)), "rrnco_train_attention_bwd")
        else:
            ws = torch.empty(h.rrnco_train_attention_tiled_workspace_bytes(n_inst, L, N), dtype=torch.uint8, device=dev)
            _check(h.rrnco_train_attention_tiled_bwd(n_inst, L, N, _p(q), _p(k), _p(v), _p(m8), _p(out), ctx.add_residual, _p(lse),
                                                     _p(d_out), _p(ws), _p(dq), _p(dk), _p(dv), _stream(dev)),
                   "rrnco_train_attention_tiled_bwd")
        return dq, dk, dv, None, None


def fused_attention(q, k, v, mask, add_residual: bool = True):
    """softmax(q_h k_h^T / 4 + mask) v_h (+ q): q [n_inst, L, 128], k / v [n_inst, N, 128], mask [n_inst, L, N] bool.
    N <= 102: K, V, dK and dV of an instance resident in shared memory; 102 < N <= 1024: the key-tiled kernels."""
    return _FusedAttention.apply(q, k, v, mask, add_residual)


class _ContextQuery(torch.autograd.Function):
    @staticmethod
    @_on_device
    def forward(ctx, table_a, index_a, table_b, index_b, state, state_w):
        h, dev = lib(), table_a.device
        n_inst, N, _ = table_a.shape
        L = index_a.shape[1]
        table_a = table_a.detach().contiguous().float()
        table_b = table_b.detach().contiguous().float() if table_b is not None else None
        index_a = index_a.contiguous()
        index_b = index_b.contiguous() if index_b is not None else None
        n_state = 0 if state is None else state.shape[-1]
        state = state.detach().contiguous().float() if state is not None else None
        state_w = state_w.detach().contiguous().float() if state_w is not None else None
        q = torch.empty(n_inst, L, 128, dtype=torch.float32, device=dev)
        _check(h.rrnco_train_context_query_fwd(n_inst * L, L, N, _p(table_a), _p(index_a), _p(table_b), _p(index_b), _p(state), n_state,
                                               _p(state_w), _p(q), _stream(dev)), "rrnco_train_context_query_fwd")
        ctx.save_for_backward(index_a, index_b, state)
        ctx.dims = (n_inst, N, L, n_state)
        return q

    @staticmethod
    @_on_device
    def backward(ctx, dq):
        index_a, index_b, state = ctx.saved_tensors
        h, dev = lib(), dq.device
        n_inst, N, L, n_state = ctx.dims
        dq = dq.contiguous().float()
        da = torch.zeros(n_inst, N, 128, dtype=torch.float32, device=dev)
        db = torch.zeros(n_inst, N, 128, dtype=torch.float32, device=dev) if index_b is not None else None
        dw = torch.zeros(n_state, 128, dtype=torch.float32, device=dev) if n_state else None
        _check(h.rrnco_train_context_query_bwd(n_inst * L, L, N, _p(dq), _p(index_a), _p(index_b), _p(state), n_state, _p(da), _p(db),
                                               _p(dw), _stream(dev)), "rrnco_train_context_query_bwd")
        return da, None, db, None, None, dw


def context_query(table_a, index_a, table_b=None, index_b=None, state=None, state_w=None):
    """q [n_inst, L, 128] = table_a[b, index_a] (+ table_b[b, index_b]) + state @ state_w; tables [n_inst, N, 128] = row_emb W_t^T,
    indices [n_inst, L] int64, state [n_inst, L, k], state_w [k, 128] (context.py:18-70 with the linear projection pulled through the gather)."""
    return _ContextQuery.apply(table_a, index_a, table_b, index_b, state, state_w)


def score_width(N: int) -> int:
    """Row width ldz of the pointer scores of an N-node instance: 128 ceil(N / 128) (one 128-column block per weight tile)."""
    return 128 * ((N + 127) // 128)


def _inst_pack(lk, transpose, dev):
    h, st = lib(), status_word(dev)
    n_inst, N, _ = lk.shape
    if N <= MAX_NODES_POINTER:
        packed = torch.empty(h.rrnco_train_inst_packed_bytes(n_inst), dtype=torch.uint8, device=dev)
        _check(h.rrnco_train_inst_pack(n_inst, N, _p(lk), transpose, _p(packed), _p(st), _stream(dev)), "rrnco_train_inst_pack")
    else:
        packed = torch.empty(h.rrnco_train_inst_tiled_packed_bytes(n_inst, N), dtype=torch.uint8, device=dev)
        _check(h.rrnco_train_inst_tiled_pack(n_inst, N, _p(lk), transpose, _p(packed), _p(st), _stream(dev)),
               "rrnco_train_inst_tiled_pack")
    return packed


def _inst_gemm(x, packed, N, transpose, a_scale, row_scale, y):
    """y = x B_b per instance: the 128-node kernel, or the key-tiled one (transpose: which operand holds the key tiles)."""
    h, dev = lib(), x.device
    n_inst, L, _ = x.shape
    st = status_word(dev)
    if N <= MAX_NODES_POINTER:
        _check(h.rrnco_train_inst_gemm(n_inst, L, _p(x), _p(packed), _p(a_scale), _p(row_scale), _p(y), _p(st), _stream(dev)),
               "rrnco_train_inst_gemm")
    else:
        _check(h.rrnco_train_inst_tiled_gemm(n_inst, L, N, transpose, _p(x), _p(packed), _p(a_scale), _p(row_scale), _p(y), _p(st),
                                             _stream(dev)), "rrnco_train_inst_tiled_gemm")


def _inst_xty(x, g, N, s_x, row_scale, dlk):
    h, dev = lib(), g.device
    n_inst, L, _ = g.shape
    st = status_word(dev)
    xty = h.rrnco_train_inst_xty if N <= MAX_NODES_POINTER else h.rrnco_train_inst_tiled_xty
    _check(xty(n_inst, L, N, _p(x), _p(g), _p(s_x), None, _p(row_scale), _p(dlk), _p(st), _stream(dev)), "rrnco_train_inst_xty")


class _PointerScores(torch.autograd.Function):
    @staticmethod
    @_on_device
    def forward(ctx, g, lk):
        dev = g.device
        g, lk = g.detach().contiguous().float(), lk.detach().contiguous().float()
        n_inst, L, _ = g.shape
        N = lk.shape[1]
        packed = _inst_pack(lk, 0, dev)
        z = torch.empty(n_inst, L, score_width(N), dtype=torch.float32, device=dev)
        _inst_gemm(g, packed, N, 0, None, None, z)
        ctx.save_for_backward(g, lk)
        return z

    @staticmethod
    @_on_device
    def backward(ctx, dz):
        g, lk = ctx.saved_tensors
        dev = g.device
        N = lk.shape[1]
        dz = dz.contiguous().float()
        s_dz = pow2_scale(dz)
        packed = _inst_pack(lk, 1, dev)
        dg = torch.empty_like(g)
        _inst_gemm(dz, packed, N, 1, s_dz, None, dg)
        dlk = torch.zeros_like(lk)
        _inst_xty(dz, g, N, s_dz, None, dlk)
        return dg, dlk


def pointer_scores(g, lk):
    """z [n_inst, L, ldz] = g lk^T (columns >= N are zero; ldz = score_width(N) = 128 ceil(N / 128)): g [n_inst, L, 128],
    lk [n_inst, N <= 1024, 128]; forward, dg and dlk on tcgen05 in the fp32-faithful fp16 hi|lo split (decoder.py:298-301 without the
    1 / sqrt(E), which the tail applies).  N <= 128: one weight tile per instance; above: ceil(N / 128) key tiles."""
    return _PointerScores.apply(g, lk)


class _LogitsTail(torch.autograd.Function):
    @staticmethod
    @_on_device
    def forward(ctx, z, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature):
        h, dev = lib(), z.device
        n_inst, L, ldz = z.shape      # N <= ldz <= 1024: the score_width(N)-wide rows of pointer_scores, or exactly N
        N = distance.shape[-1]
        jac = z.detach()
        if not jac.is_contiguous() or jac.dtype != torch.float32:
            jac = jac.contiguous().float()
        rows = n_inst * L
        logp = torch.empty(n_inst, L, dtype=torch.float32, device=dev)
        da = torch.empty(n_inst, L, dtype=torch.float32, device=dev)
        db = torch.empty(n_inst, L, dtype=torch.float32, device=dev) if duration is not None else None
        alpha_d = alpha.detach().reshape(-1).float().contiguous()
        beta_d = beta.detach().reshape(-1).float().contiguous() if duration is not None else None
        # every argument stays referenced until the launch is enqueued (a temporary's block could be handed to the next one)
        distance, cur, act = distance.contiguous(), cur.contiguous(), act.contiguous()
        duration = duration.contiguous() if duration is not None else None
        m8 = mask.contiguous().view(torch.uint8)
        _check(h.rrnco_train_logits_tail(rows, L, N, ldz, _p(jac), _p(distance), _p(duration), _p(cur), _p(m8), _p(act), _p(alpha_d), _p(beta_d),
                                         1.0 / math.sqrt(128.0), float(tanh_clipping), float(temperature), _p(logp), _p(da), _p(db),
                                         _stream(dev)), "rrnco_train_logits_tail")
        ctx.save_for_backward(jac, da, db)
        ctx.shapes = (alpha.shape, beta.shape if beta is not None else None)
        return logp

    @staticmethod
    @_on_device
    def backward(ctx, g):
        jac, da, db = ctx.saved_tensors
        g = g.float()
        dz = jac.mul_(g.unsqueeze(-1))  # the Jacobian is this node's own buffer (the raw scores were overwritten in place)
        dalpha = (g * da).sum().reshape(ctx.shapes[0])
        dbeta = (g * db).sum().reshape(ctx.shapes[1]) if db is not None else None
        return dz, dalpha, dbeta, None, None, None, None, None, None, None


def fused_logits_tail(z, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature):
    """log pi(act | state) [n_inst, L] from the raw pointer scores z = g . Lk^T [n_inst, L, ldz], N <= ldz <= 1024 (consumed:
    overwritten in place by the Jacobian); distance / duration [n_inst, N, N], cur / act [n_inst, L] int64, mask [n_inst, L, N] bool."""
    return _LogitsTail.apply(z, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature)


class _PointerLogProb(torch.autograd.Function):
    """pointer_scores + fused_logits_tail as ONE node: the backward pass feeds the saved Jacobian and the upstream gradient of
    each row straight into the dg / dlk kernels (`row_scale`), so dz = g_row J is never written."""

    @staticmethod
    @_on_device
    def forward(ctx, g, lk, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature):
        h, dev = lib(), g.device
        g, lk = g.detach().contiguous().float(), lk.detach().contiguous().float()
        n_inst, L, _ = g.shape
        N = lk.shape[1]
        ldz = score_width(N)
        packed = _inst_pack(lk, 0, dev)
        jac = torch.empty(n_inst, L, ldz, dtype=torch.float32, device=dev)
        _inst_gemm(g, packed, N, 0, None, None, jac)
        logp = torch.empty(n_inst, L, dtype=torch.float32, device=dev)
        da = torch.empty(n_inst, L, dtype=torch.float32, device=dev)
        db = torch.empty(n_inst, L, dtype=torch.float32, device=dev) if duration is not None else None
        alpha_d = alpha.detach().reshape(-1).float().contiguous()
        beta_d = beta.detach().reshape(-1).float().contiguous() if duration is not None else None
        distance, cur, act = distance.contiguous(), cur.contiguous(), act.contiguous()
        duration = duration.contiguous() if duration is not None else None
        m8 = mask.contiguous().view(torch.uint8)
        _check(h.rrnco_train_logits_tail(n_inst * L, L, N, ldz, _p(jac), _p(distance), _p(duration), _p(cur), _p(m8), _p(act),
                                         _p(alpha_d), _p(beta_d), 1.0 / math.sqrt(128.0), float(tanh_clipping), float(temperature),
                                         _p(logp), _p(da), _p(db), _stream(dev)), "rrnco_train_logits_tail")
        ctx.save_for_backward(g, lk, jac, da, db)
        ctx.shapes = (alpha.shape, beta.shape if beta is not None else None)
        # |J| <= clip / (T sqrt(E)) (tanh' <= 1, exp / (exp + 1e-6) <= 1, |delta - softmax| <= 1): bound of the scaled operand
        ctx.jmax = (float(tanh_clipping) if tanh_clipping > 0 else 1.0) / (float(temperature) * math.sqrt(128.0))
        return logp

    @staticmethod
    @_on_device
    def backward(ctx, gl):
        g, lk, jac, da, db = ctx.saved_tensors
        dev = g.device
        N = lk.shape[1]
        gl = gl.contiguous().float()
        s_dz = pow2_scale(gl, bound_factor=ctx.jmax)
        packed = _inst_pack(lk, 1, dev)
        dg = torch.empty_like(g)
        _inst_gemm(jac, packed, N, 1, s_dz, gl, dg)
        dlk = torch.zeros_like(lk)
        _inst_xty(jac, g, N, s_dz, gl, dlk)
        dalpha = (gl * da).sum().reshape(ctx.shapes[0])
        dbeta = (gl * db).sum().reshape(ctx.shapes[1]) if db is not None else None
        return dg, dlk, dalpha, dbeta, None, None, None, None, None, None, None


def pointer_logprob(g, lk, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature):
    """log pi(act | state) [n_inst, L] from the pointer input g [n_inst, L, 128] and the logit keys lk [n_inst, N <= 1024, 128]
    (decoder.py:183-198, 298-301; decoding.py:311-399): pointer_scores and fused_logits_tail as one autograd node.  The saved
    Jacobian is [n_inst, L, score_width(N)]."""
    return _PointerLogProb.apply(g, lk, alpha, beta, distance, duration, cur, mask, act, tanh_clipping, temperature)
