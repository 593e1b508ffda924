"""ctypes binding of librrnco_b200.so (include/rrnco_b200.h).

The product path has NO CPU fallback: if the shared library is missing or a call is made without a CUDA
tensor, this module raises.  Torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librrnco_b200.so")

ENV_ID = {"atsp": 0, "rcvrp": 1, "rcvrptw": 2}
DECODE_ID = {"greedy": 0, "sampling": 1, "evaluate": 2}
DEV_NAN_LOGITS, DEV_INFEASIBLE, DEV_NO_FEASIBLE, DEV_TRUNCATED, DEV_SOFTMAX_RANGE = 1, 2, 4, 8, 16
DEV_BAD_PARENT = 32
MAX_NODES_TILE = 128     # one key tile: rrnco_decoder_logits, single-tile fused kernels
MAX_NODES_FUSED = 1024   # rrnco_rollout (key-tiled kernel above MAX_NODES_TILE)
MAX_BEAM_WIDTH = 1024   # rrnco_beam_select
MIN_STARTS_TILED = 8   # RRNetDecoder.forward: starts per instance from which the any-N tile kernels serve every N

_f = C.c_void_p  # every device pointer travels as void*


class DecoderWeights(C.Structure):
    _fields_ = [("ffn_w1", _f), ("ffn_b1", _f), ("ffn_w2", _f), ("ffn_b2", _f), ("ctx_state_w", _f),
                ("ctx_placeholder_q", _f), ("alpha", C.c_float), ("beta", C.c_float),
                ("tanh_clipping", C.c_float), ("temperature", C.c_float)]


class DecoderCache(C.Structure):
    _fields_ = [("glimpse_key", _f), ("glimpse_val", _f), ("logit_key", _f), ("ctx_node_proj", _f),
                ("ctx_node_proj2", _f)]


class InstanceData(C.Structure):
    _fields_ = [("data_rows", C.c_int64), ("distance", _f), ("duration", _f), ("demand", _f),
                ("demand_backhaul", _f), ("time_windows", _f), ("service_time", _f), ("vehicle_capacity", _f),
                ("distance_limit", _f), ("open_route", _f), ("backhaul_class", _f), ("min_distance", _f),
                ("max_distance", _f)]


class RmtvrpState(C.Structure):
    _fields_ = [("current_node", _f), ("current_time", _f), ("current_route_length", _f),
                ("used_capacity_linehaul", _f), ("used_capacity_backhaul", _f), ("visited", _f)]


_SIGNATURES = {
    "rrnco_abi_version": (C.c_int, []),
    "rrnco_strerror": (C.c_char_p, [C.c_int]),
    "rrnco_u01": (C.c_float, [C.c_uint32]),
    "rrnco_set_precision": (C.c_int, [C.c_int32]),
    "rrnco_set_ffn_engine": (C.c_int, [C.c_int32]),
    "rrnco_set_step_tiling": (C.c_int, [C.c_int32]),
    "rrnco_set_start_split": (C.c_int, [C.c_int32]),
    "rrnco_nab_packed_floats": (C.c_int64, []),
    "rrnco_nab_pack": (C.c_int, [_f] * 14),
    "rrnco_nab_dur_packed_bytes": (C.c_int64, []),
    "rrnco_nab_dur_pack": (C.c_int, [_f, _f, _f, _f]),
    "rrnco_nab_dur_gating": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, C.c_int32, _f, C.c_float, _f, _f, _f]),
    "rrnco_aft_nab": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, _f, _f, C.c_int32, _f, C.c_float, _f, _f]),
    "rrnco_nab_gating": (C.c_int, [C.c_int64, C.c_int32, _f, _f, C.c_int32, _f, C.c_float, C.c_int32, _f, _f]),
    "rrnco_rollout_tile_rows": (C.c_int32, [C.c_int32, C.c_int32, C.c_int64, C.c_int32]),
    "rrnco_minmax_normalize": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, _f, _f]),
    "rrnco_gather_submatrix": (C.c_int, [_f, C.c_int32, _f, C.c_int64, C.c_int32, _f, C.c_int32, _f, _f, _f]),
    "rrnco_gather_submatrix_f32": (C.c_int, [_f, C.c_int32, _f, C.c_int64, C.c_int32, _f, C.c_int32, _f, _f, _f]),
    "rrnco_city_matrix_to_f32": (C.c_int, [_f, C.c_int64, _f, _f]),
    "rrnco_atsp_step": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_rcvrp_step": (C.c_int, [C.c_int64, C.c_int32, C.c_int64, _f, _f, _f, C.c_int64, _f, _f, _f, _f, _f,
                                   _f, _f, _f, _f]),
    "rrnco_rmtvrp_step": (C.c_int, [C.c_int64, C.c_int32, C.POINTER(InstanceData), _f, C.POINTER(RmtvrpState),
                                    C.POINTER(RmtvrpState), _f, _f, _f]),
    "rrnco_tour_reward": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int64, _f, _f, C.c_int32, _f, _f, _f,
                                    _f, _f, _f]),
    "rrnco_precompute_cache": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, _f, _f, _f, _f, C.c_int32, _f, _f, _f,
                                         _f, _f, _f]),
    "rrnco_decoder_logits": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.POINTER(DecoderWeights),
                                       C.POINTER(DecoderCache), C.POINTER(InstanceData), _f, _f, _f, _f, C.c_int32,
                                       _f, _f, _f]),
    "rrnco_decoder_logits_large_workspace_bytes": (C.c_int64, [C.c_int64]),
    "rrnco_decoder_logits_large": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.POINTER(DecoderWeights),
                                             C.POINTER(DecoderCache), C.POINTER(InstanceData), _f, _f, _f, _f,
                                             C.c_int32, _f, _f, _f, _f]),
    "rrnco_select_action": (C.c_int, [C.c_int64, C.c_int32, _f, _f, C.c_int32, C.c_float, C.c_float, C.c_uint64,
                                      C.c_int32, _f, _f, _f, _f, _f]),
    "rrnco_select_action_filtered": (C.c_int, [C.c_int64, C.c_int32, _f, _f, C.c_int32, C.c_float, C.c_float, C.c_uint64,
                                               C.c_int32, _f, _f, _f, _f, C.c_int32, C.c_float, _f]),
    "rrnco_beam_select": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _f, _f, _f, C.c_float, C.c_float, _f, _f, _f, _f, _f,
                                    _f]),
    "rrnco_beam_backtrack": (C.c_int, [C.c_int64, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_pointer_ffn_workspace_bytes": (C.c_int64, []),
    "rrnco_pointer_ffn": (C.c_int, [C.c_int64, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_rollout_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int64, C.c_int32]),
    "rrnco_rollout": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                C.POINTER(DecoderWeights), C.POINTER(DecoderCache), C.POINTER(InstanceData), _f,
                                C.c_int32, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f, _f]),
    "rrnco_rollout_filtered": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                         C.POINTER(DecoderWeights), C.POINTER(DecoderCache), C.POINTER(InstanceData), _f,
                                         C.c_int32, C.c_int32, _f, _f, _f, _f, _f, _f, _f, _f, C.c_int32, C.c_float, _f]),
}

_lib = None
launch_count = 0  # library calls that enqueued work
kernel_count = 0  # CUDA kernels those calls launched (bench.py reports it as gpu_launches)
_KERNELS_PER_CALL = {"rrnco_rollout": 3, "rrnco_rollout_filtered": 3, "rrnco_pointer_ffn": 2, "rrnco_decoder_logits_large": 4}  # rollout: weight pack + rollout + finalize  # rollout_kernel + finalize_kernel; every other entry point launches one


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m rrnco_b200.build` (or __graft_entry__.build()). "
                "rrnco_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def exported_symbols():
    return list(_SIGNATURES)


class RRNCOError(RuntimeError):
    pass


def check(code: int):
    if code != 0:
        raise RRNCOError(f"librrnco_b200: {lib().rrnco_strerror(code).decode()} (code {code})")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL). Refuses host tensors: there is no CPU path."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RRNCOError("rrnco_b200 needs CUDA tensors (no CPU fallback); got a tensor on " + str(t.device))
    if not t.is_contiguous():
        raise RRNCOError("rrnco_b200 needs contiguous tensors")
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def call(name, *args):
    global launch_count, kernel_count
    launch_count += 1
    kernel_count += _KERNELS_PER_CALL.get(name, 1)
    check(getattr(lib(), name)(*args))


def count_call(name: str):
    """Launch accounting for calls that do not go through `call` (the torch-op binding)."""
    global launch_count, kernel_count
    launch_count += 1
    kernel_count += _KERNELS_PER_CALL.get(name, 1)


def set_precision(passes: int):
    check(lib().rrnco_set_precision(passes))


def set_step_tiling(mode):
    """Any-N per-step decoder: 1 / True = shared-memory key tiles per (instance, start group) with tensor-core logits
    (default), 2 = same tiling with FFMA logits, 0 / False = per-rollout streaming."""
    check(lib().rrnco_set_step_tiling(int(mode)))


def set_ffn_engine(engine: int):
    """Engine of the fused rollout kernel: 2 = lean kernel for N <= 112, else the one-CTA tcgen05 kernel (default), 1 = one-CTA
    tcgen05 kernel, 0 = mma.sync FFN."""
    check(lib().rrnco_set_ffn_engine(engine))


def raise_device_status(word: int):
    """Surface the sticky device status with the reference's exception texts."""
    if word & DEV_TRUNCATED:  # rrnco/models/policy.py:222-226 logs an error and breaks; so does this
        import logging
        logging.getLogger("rrnco_b200").error("Exceeded maximum number of steps during decoding: rollouts that had "
                                              "not finished were cut and scored as they stood")
    if word & DEV_NAN_LOGITS:
        raise AssertionError("Logits contain NaNs")  # rrnco/models/decoder.py:303-304
    if word & DEV_INFEASIBLE:
        raise AssertionError("infeasible action selected")  # rrnco/models/decoding.py:278-280
    if word & DEV_NO_FEASIBLE:
        raise AssertionError("no feasible action (fully masked row)")
    if word & DEV_BAD_PARENT:
        raise AssertionError("beam backtrack: a parent row outside the beam rows (corrupted beam records)")
