"""Drop-in decoder / policy: the reference's `RRNetDecoder` and `RRNetPolicy` call surface with the per-step
decoder and the whole decode loop running as fused sm_100a kernels (librrnco_b200).

  RRNetDecoder  <- rrnco/models/decoder.py:46-232 (+ RRNet_PointerAttention :235-329); parameter names are
                   identical, so reference checkpoints load with `load_state_dict`.
  RRNetPolicy   <- rrnco/models/policy.py:19-255; `forward` returns the same out-dict.  The encoder stays the
                   reference's PyTorch module (pass it as `encoder=`), as BASELINE.json's north star states.

The logit filters `top_k` / `top_p` of rl4co's `process_logits` run inside the decode kernels (any decode type), except
under grad in phase "train" without forced actions: the differentiable replay does not filter, so that call raises.
`decode_type="beam_search"` (rl4co BeamSearch; `beam_width=`, `select_best=` which defaults to True there) runs in one
launch of the lean rollout kernel (rrnco_beam_rollout) for N <= 112 and up to 128 beams under the default engine and
precision, and on the per-step kernel pipeline otherwise (rrnco_beam_select picks the beams); rrnco_beam_backtrack aligns
the sequences.  It raises NotImplementedError together with top_k / top_p, with `actions=`, and under grad in phase "train".
`select_best=True` on a multistart greedy / sampling decode keeps each instance's best start (first maximum of the reward).
Unsupported reference options raise NotImplementedError (store_all_logp / return_entropy, mask_logits=False, dynamic
embeddings): they are not on any BASELINE config.
"""
from __future__ import annotations

import os

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple, Union

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib
from ._lib import DECODE_ID, ENV_ID, DecoderCache, DecoderWeights, InstanceData, call, ptr, stream_ptr
from .envs import _u8, tour_reward

CTX_IN = {"atsp": 256, "rcvrp": 129, "rcvrptw": 132}
N_STATE = {"atsp": 0, "rcvrp": 1, "rcvrptw": 4}


@dataclass
class PrecomputedCache:
    """decoder.py:25-43, plus the node half of the context projection the fused kernels consume."""
    node_embeddings: Tensor
    graph_context: Union[Tensor, float]
    glimpse_key: Tensor
    glimpse_val: Tensor
    logit_key: Tensor
    ctx_node_proj: Optional[Tensor] = None
    ctx_node_proj2: Optional[Tensor] = None

    def struct(self) -> DecoderCache:
        c = DecoderCache()
        c.glimpse_key, c.glimpse_val, c.logit_key = ptr(self.glimpse_key), ptr(self.glimpse_val), ptr(self.logit_key)
        c.ctx_node_proj, c.ctx_node_proj2 = ptr(self.ctx_node_proj), ptr(self.ctx_node_proj2)
        return c


class _Context(nn.Module):
    """Parameter holder named like rl4co's EnvContext (project_context [+ W_placeholder for atsp])."""

    def __init__(self, env_name, embed_dim):
        super().__init__()
        self.project_context = nn.Linear(CTX_IN[env_name], embed_dim, bias=False)
        if env_name == "atsp":
            self.W_placeholder = nn.Parameter(torch.Tensor(2 * embed_dim).uniform_(-1, 1))


class _FFN(nn.Module):
    def __init__(self, embed_dim):
        super().__init__()
        self.lins = nn.ModuleList([nn.Linear(embed_dim, 4 * embed_dim), nn.Linear(4 * embed_dim, embed_dim)])


class _Pointer(nn.Module):
    def __init__(self, embed_dim):
        super().__init__()
        self.project_out = nn.Linear(embed_dim, embed_dim, bias=False)  # unused upstream too (decoder.py:295)
        self.ffn = _FFN(embed_dim)


def instance_tensors_from_td(env_name: str, td) -> list:
    """The members of rrnco_instance_data_t as a list of (optional) tensors, in order (torch-op binding)."""
    f = lambda t: t.to(torch.float32).contiguous()
    k = td.keys()
    d = [None] * 12
    d[0] = f(td["distance_matrix"])
    if "min_distance" in k:
        d[10], d[11] = f(td["min_distance"]), f(td["max_distance"])
    if env_name == "rcvrp":
        d[2], d[6] = f(td["demand"]), f(td["vehicle_capacity"].reshape(-1))
    elif env_name == "rcvrptw":
        d[1], d[2], d[3] = f(td["duration_matrix"]), f(td["demand_linehaul"]), f(td["demand_backhaul"])
        d[4], d[5], d[6] = f(td["time_windows"]), f(td["service_time"]), f(td["vehicle_capacity"].reshape(-1))
        d[7], d[8], d[9] = f(td["distance_limit"].reshape(-1)), _u8(td["open_route"].reshape(-1)), f(td["backhaul_class"].reshape(-1))
    return d


def instance_data_from_td(env_name: str, td, keep: list) -> InstanceData:
    """InstanceData over a reset td; rows are indexed by instance (b % data_rows)."""
    def put(t, dtype=torch.float32):
        t = _u8(t) if dtype == torch.uint8 else t.to(dtype).contiguous()
        keep.append(t)
        return ptr(t)

    d = InstanceData()
    d.data_rows = td["distance_matrix"].shape[0]
    d.distance = put(td["distance_matrix"])
    if "min_distance" in td.keys():
        d.min_distance, d.max_distance = put(td["min_distance"]), put(td["max_distance"])
    if env_name == "rcvrp":
        d.demand = put(td["demand"])
        d.vehicle_capacity = put(td["vehicle_capacity"].reshape(-1))
    elif env_name == "rcvrptw":
        d.duration = put(td["duration_matrix"])
        d.demand = put(td["demand_linehaul"])
        d.demand_backhaul = put(td["demand_backhaul"])
        d.time_windows = put(td["time_windows"])
        d.service_time = put(td["service_time"])
        d.vehicle_capacity = put(td["vehicle_capacity"].reshape(-1))
        d.distance_limit = put(td["distance_limit"].reshape(-1))
        d.open_route = put(td["open_route"].reshape(-1), torch.uint8)
        d.backhaul_class = put(td["backhaul_class"].reshape(-1))
    return d


class RRNetDecoder(nn.Module):
    def __init__(self, embed_dim: int = 128, num_heads: int = 8, env_name: str = "rcvrp", mask_inner: bool = True,
                 out_bias_pointer_attn: bool = False, linear_bias: bool = False, use_graph_context: bool = True,
                 check_nan: bool = True, **unused):
        super().__init__()
        env_name = getattr(env_name, "name", env_name)
        if env_name not in ENV_ID:
            raise ValueError(f"Unknown environment name '{env_name}'. Available: {list(ENV_ID)}")
        if embed_dim != 128 or num_heads != 8:
            raise NotImplementedError("the fused kernels are built for embed_dim 128, 8 heads (experiment/rrnet.yaml)")
        if not mask_inner or out_bias_pointer_attn or linear_bias:
            raise NotImplementedError("mask_inner=False / pointer or linear biases are not on the reference's configs")
        self.env_name, self.embed_dim, self.num_heads = env_name, embed_dim, num_heads
        self.check_nan = check_nan
        if env_name == "rcvrptw":
            self.beta = nn.Parameter(torch.tensor([1.0]))
        self.context_embedding = _Context(env_name, embed_dim)
        self.pointer = _Pointer(embed_dim)
        self.project_node_embeddings = nn.Linear(embed_dim, 3 * embed_dim, bias=False)
        self.project_fixed_context = nn.Linear(embed_dim, embed_dim, bias=False)  # unused: graph_context = 0
        self.alpha = nn.Parameter(torch.tensor([1.0]))
        self.is_dynamic_embedding = False
        self._wcache = None

    # -- weights handed to the kernels ---------------------------------------------------------------
    def kernel_weight_tensors(self):
        """The members of rrnco_decoder_weights_t as tensors, in order (torch-op binding); (alpha, beta) as floats."""
        E = self.embed_dim
        f = lambda t: t.detach().to(torch.float32).contiguous()
        lins = self.pointer.ffn.lins
        wc = self.context_embedding.project_context.weight.detach().float()
        state_w = f(wc[:, E:].t()) if self.env_name != "atsp" else None
        placeholder = f(wc @ self.context_embedding.W_placeholder.detach().float()) if self.env_name == "atsp" else None
        w, _ = self.kernel_weights()
        return [f(lins[0].weight), f(lins[0].bias), f(lins[1].weight), f(lins[1].bias), state_w, placeholder], w.alpha, w.beta

    def kernel_weights(self, temperature: float = 1.0, tanh_clipping: float = 10.0):
        """(DecoderWeights struct, keep-alive list)."""
        E = self.embed_dim
        keep = []
        w = DecoderWeights()

        def put(t):
            t = t.detach().to(torch.float32).contiguous()
            keep.append(t)
            return ptr(t)

        lins = self.pointer.ffn.lins
        w.ffn_w1, w.ffn_b1, w.ffn_w2, w.ffn_b2 = put(lins[0].weight), put(lins[0].bias), put(lins[1].weight), put(lins[1].bias)
        wc = self.context_embedding.project_context.weight.detach().float()
        if self.env_name != "atsp":
            w.ctx_state_w = put(wc[:, E:].t())  # [n_state, E]
        else:
            w.ctx_placeholder_q = put(wc @ self.context_embedding.W_placeholder.detach().float())
        beta = self.beta if self.env_name == "rcvrptw" else self.alpha
        key = (self.alpha._version, beta._version, self.alpha.data_ptr())
        if self._wcache is None or self._wcache[0] != key:  # one D2H read per parameter update, not per call
            self._wcache = (key, torch.stack([self.alpha.detach().float().reshape(()),
                                              beta.detach().float().reshape(())]).tolist())
        w.alpha, w.beta = self._wcache[1]
        w.tanh_clipping, w.temperature = float(tanh_clipping), float(temperature)
        return w, keep

    # -- reference API ---------------------------------------------------------------------------------
    def _precompute_cache(self, embeddings: Tuple[Tensor, Tensor], num_starts: int = 0) -> PrecomputedCache:
        row_emb, col_emb = embeddings
        row_emb, col_emb = row_emb.float().contiguous(), col_emb.float().contiguous()
        B, N, E = col_emb.shape
        outs = [torch.empty_like(col_emb) for _ in range(4)]
        p2 = torch.empty_like(col_emb) if self.env_name == "atsp" else None
        wn = self.project_node_embeddings.weight.detach().float().contiguous()
        wc = self.context_embedding.project_context.weight.detach().float().contiguous()
        call("rrnco_precompute_cache", ENV_ID[self.env_name], B, N, ptr(row_emb), ptr(col_emb), ptr(wn), ptr(wc),
             wc.shape[1], ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), ptr(p2), stream_ptr(col_emb.device))
        return PrecomputedCache(node_embeddings=row_emb, graph_context=0, glimpse_key=outs[0], glimpse_val=outs[1],
                                logit_key=outs[2], ctx_node_proj=outs[3], ctx_node_proj2=p2)

    def pre_decoder_hook(self, td, env, embeddings, num_starts: int = 0):
        return td, env, self._precompute_cache(embeddings, num_starts=num_starts)

    def _ctx_state(self, td):
        if self.env_name == "rcvrp":
            return (td["vehicle_capacity"] - td["used_capacity"]).float()
        used = torch.where(td["used_capacity_backhaul"] == 0, td["used_capacity_linehaul"], td["used_capacity_backhaul"])
        rem = torch.nan_to_num(td["distance_limit"] - td["current_route_length"], posinf=10)
        return torch.cat((td["vehicle_capacity"] - used, td["current_time"], td["open_route"].float(), rem), -1).float()

    def forward(self, td, cached: PrecomputedCache, num_starts: int = 0) -> Tuple[Tensor, Tensor]:
        """One decode step: (logits [R,N] fp32 after the distance/duration bias, mask [R,N] bool)."""
        mask = td["action_mask"].contiguous()
        R, N = mask.shape
        S = num_starts if num_starts > 1 else 1
        n_inst = R // S
        if cached.glimpse_key.shape[0] != n_inst:
            raise ValueError(f"cache holds {cached.glimpse_key.shape[0]} instances, td implies {n_inst}")
        keep = []
        w, keep_w = self.kernel_weights()
        data = InstanceData()  # the logits kernel only needs the matrices (bias rows)
        data.data_rows = td["distance_matrix"].shape[0]
        dm = td["distance_matrix"].float().contiguous()
        keep.append(dm)
        data.distance = ptr(dm)
        if self.env_name == "rcvrptw":
            du = td["duration_matrix"].float().contiguous()
            keep.append(du)
            data.duration = ptr(du)
        cur = td["current_node"].reshape(-1).contiguous()
        first, state, placeholder = None, None, 0
        if self.env_name == "atsp":
            first = td["first_node"].reshape(-1).contiguous()
            if S == 1:  # only reachable without multistart; upstream syncs here too (TSPContext .item())
                placeholder = int(int(td["i"].reshape(-1)[0]) < 1)
        else:
            state = self._ctx_state(td).contiguous()
        logits = torch.empty((R, N), dtype=torch.float32, device=mask.device)
        status = torch.zeros(1, dtype=torch.int32, device=mask.device)
        cs = cached.struct()
        # per-step kernels: with >= 8 starts per instance the key-sharing tile kernels (any N) are also the faster ones at
        # N <= 128 (RCVRP n=100 x8 aug x101 starts, per-step loop: 904 vs 661 instances/s, tools/per_step_probe.py)
        if N <= _lib.MAX_NODES_TILE and S < _lib.MIN_STARTS_TILED:
            call("rrnco_decoder_logits", ENV_ID[self.env_name], N, n_inst, S, C.byref(w), C.byref(cs), C.byref(data),
                 ptr(cur), ptr(first), ptr(_u8(mask)), ptr(state), placeholder, ptr(logits), ptr(status),
                 stream_ptr(mask.device))
        else:  # key-streaming kernels: any N
            ws = torch.empty(_lib.lib().rrnco_decoder_logits_large_workspace_bytes(R), dtype=torch.uint8,
                             device=mask.device)
            call("rrnco_decoder_logits_large", ENV_ID[self.env_name], N, n_inst, S, C.byref(w), C.byref(cs),
                 C.byref(data), ptr(cur), ptr(first), ptr(_u8(mask)), ptr(state), placeholder, ptr(logits),
                 ptr(status), ptr(ws), stream_ptr(mask.device))
        if self.check_nan:  # upstream asserts (and syncs) every step: decoder.py:303-304
            _lib.raise_device_status(int(status.item()) & _lib.DEV_NAN_LOGITS)
        return logits, mask


class RRNetPolicy(nn.Module):
    def __init__(self, encoder: nn.Module = None, decoder: nn.Module = None, embed_dim: int = 128,
                 num_heads: int = 8, env_name: str = "rcvrp", temperature: float = 1.0, tanh_clipping: float = 10.0,
                 mask_logits: bool = True, train_decode_type: str = "sampling", val_decode_type: str = "greedy",
                 test_decode_type: str = "greedy", check_nan: bool = True, **unused_kwargs):
        super().__init__()
        env_name = getattr(env_name, "name", env_name)
        if encoder is None:
            raise ValueError("pass the reference's RRNetEncoder (or any module returning (row_emb, col_emb)) as "
                             "`encoder=`: the encoder stays in the reference PyTorch path")
        if not mask_logits:
            raise NotImplementedError("mask_logits=False")
        self.encoder = encoder
        self.decoder = decoder if decoder is not None else RRNetDecoder(embed_dim, num_heads, env_name, check_nan=check_nan)
        self.env_name = env_name
        self.temperature, self.tanh_clipping, self.mask_logits = temperature, tanh_clipping, mask_logits
        self.train_decode_type, self.val_decode_type, self.test_decode_type = (
            train_decode_type, val_decode_type, test_decode_type)
        self.seed = None  # sampling seed base; None = derived from torch.initial_seed() and the distributed rank
        self._calls = 0
        self.train_replay_autocast = None  # e.g. torch.bfloat16: autocast of the differentiable replay in phase "train"
        self.large_n_path = "fused"  # 128 < N <= 1024: "fused" = key-tiled rollout kernel, "stepwise" = per-step kernel pipeline

    def _seed_base(self) -> int:
        """Philox key of the Gumbel-max sampler when the caller passes no `seed=`: follows torch / Lightning seeding
        (`seed_everything` sets torch.initial_seed()) and differs per DDP rank, so ranks draw independent noise."""
        if self.seed is not None:
            return int(self.seed)
        rank = 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            rank = torch.distributed.get_rank()
        else:
            rank = int(os.environ.get("RANK", 0))
        return (torch.initial_seed() + 0x9E3779B97F4A7C15 * (rank + 1)) & (2**64 - 1)

    def forward(self, td, env=None, phase: str = "train", calc_reward: bool = True, return_actions: bool = True,
                return_entropy: bool = False, return_hidden: bool = False, return_init_embeds: bool = False,
                return_sum_log_likelihood: bool = True, actions=None, max_steps=1_000_000, **decoding_kwargs) -> dict:
        if env is None or isinstance(env, str):
            raise ValueError("pass an instantiated rrnco_b200 env")
        if return_entropy or decoding_kwargs.get("store_all_logp"):
            raise NotImplementedError("store_all_logp / return_entropy")
        top_k, top_p = filter_args(decoding_kwargs.pop("top_k", None), decoding_kwargs.pop("top_p", None))
        filtered = filter_active(top_k, top_p)
        if filtered and phase == "train" and torch.is_grad_enabled() and actions is None:
            raise NotImplementedError("top_k / top_p under grad in phase 'train': the differentiable replay of the sampled "
                                      "actions (training.batched_logprobs) does not filter")
        decode_type = decoding_kwargs.pop("decode_type", None)
        beam = decode_type == "beam_search" or (decode_type is None and actions is None
                                                and getattr(self, f"{phase}_decode_type") == "beam_search")
        select_best = decoding_kwargs.pop("select_best", None)
        select_best = beam if select_best is None else bool(select_best)  # BeamSearch defaults to True, the others to False
        beam_width = decoding_kwargs.pop("beam_width", None)
        if beam:
            if actions is not None:
                raise NotImplementedError("actions= with decode_type 'beam_search': evaluate given actions with the "
                                          "default decode type")
            if filtered:
                raise NotImplementedError("top_k / top_p with decode_type 'beam_search'")
            if phase == "train" and torch.is_grad_enabled():
                raise NotImplementedError("beam search under grad in phase 'train': the differentiable replay of the "
                                          "actions (training.batched_logprobs) does not beam")
            if beam_width is not None:
                beam_width = beam_args(beam_width)
        if td.device.type != "cuda":
            td = td.to(env.device)
        if beam and beam_width is None:
            beam_width = beam_args(env.get_num_starts(td))  # BeamSearch.pre_decoder_hook

        row_emb, col_emb = self.encoder(td, phase=phase)  # policy.py:176

        if beam:
            cache = self.decoder._precompute_cache((row_emb, col_emb), num_starts=beam_width)
            self._calls += 1
            fused = fused_beam_serves(self.env_name, cache.glimpse_key.shape[1], beam_width)
            out = (fused_beam_rollout if fused else beam_search_rollout)(self.decoder, cache, env, td, beam_width,
                                      temperature=decoding_kwargs.pop("temperature", self.temperature),
                                      tanh_clipping=decoding_kwargs.pop("tanh_clipping", self.tanh_clipping),
                                      calc_reward=calc_reward or select_best,
                                      per_step_logprobs=not return_sum_log_likelihood, check=self.decoder.check_nan)
            outdict = {"reward": out["reward"],
                       "log_likelihood": out["log_likelihood"] if return_sum_log_likelihood else out["logprobs"]}
            if "normalized_reward" in out:
                outdict["normalized_reward"] = out["normalized_reward"]
            if return_actions:
                outdict["actions"] = out["actions"]
            if select_best:
                outdict = select_best_rows(outdict, beam_width)
            if return_hidden:
                outdict["hidden"] = cache
            return outdict

        if actions is not None:
            decode_type = "evaluate"
        elif decode_type is None:
            decode_type = getattr(self, f"{phase}_decode_type")
        if decode_type.replace("multistart_", "") not in DECODE_ID:
            raise NotImplementedError(f"decode type '{decode_type}' (only greedy / sampling / evaluate [+ multistart_])")
        num_starts = decoding_kwargs.pop("num_starts", None)
        multistart = "multistart" in decode_type  # decoding.py:31-32
        if num_starts is not None:  # decoding.py:117-118
            multistart = num_starts > 1
        if multistart and num_starts is None:
            num_starts = env.get_num_starts(td)  # decoding.py:162-163
        S = num_starts if multistart else 1
        calc_reward = calc_reward or (select_best and S > 1)  # rl4co's _select_best computes the rewards it ranks by
        temperature = decoding_kwargs.pop("temperature", self.temperature)
        tanh_clipping = decoding_kwargs.pop("tanh_clipping", self.tanh_clipping)

        cache = self.decoder._precompute_cache((row_emb, col_emb), num_starts=S)
        self._calls += 1
        n_nodes = cache.glimpse_key.shape[1]
        # N <= 128: single-tile fused kernels; N <= 1024: key-tiled fused kernel; beyond (or large_n_path = "stepwise"): the
        # per-step kernel pipeline.  top-k / top-p above 128 nodes: the per-step pipeline (the key-tiled kernel never holds
        # a whole row of scores, which the filters need)
        use_fused = n_nodes <= _lib.MAX_NODES_TILE or (n_nodes <= _lib.MAX_NODES_FUSED and self.large_n_path == "fused"
                                                       and not filtered)
        rollout_fn = fused_rollout if use_fused else stepwise_rollout
        rollout_args = dict(forced_actions=actions, seed=decoding_kwargs.pop("seed", self._seed_base() + self._calls),
                            temperature=temperature, tanh_clipping=tanh_clipping, calc_reward=calc_reward,
                            per_step_logprobs=not return_sum_log_likelihood, check=self.decoder.check_nan,
                            top_k=top_k, top_p=top_p)
        try:
            out = rollout_fn(self.decoder, cache, env, td, S, multistart, decode_type.replace("multistart_", ""), **rollout_args)
        except SoftmaxRangeError:
            FALLBACKS["softmax_range"] += 1
            # key-tiled fused kernel only (N > 128): a head's scores left the range of its fixed softmax shift; the per-step
            # kernels (exact running maximum) serve such checkpoints -- still the CUDA path, never a CPU fallback
            out = stepwise_rollout(self.decoder, cache, env, td, S, multistart, decode_type.replace("multistart_", ""),
                                   **rollout_args)
        outdict = {"reward": out["reward"],
                   "log_likelihood": out["log_likelihood"] if return_sum_log_likelihood else out["logprobs"]}
        if phase == "train" and torch.is_grad_enabled() and multistart and actions is None:
            # rl.py:119-128 differentiates out["log_likelihood"]: the kernel's value carries no graph, so the sampled
            # actions are re-evaluated by the differentiable batched replay (training.py), same encoder output
            from .training import batched_logprobs, iter_decode_inputs
            inputs = iter_decode_inputs(self.decoder, env, td, out["actions"], S)   # generator: replay overlaps the kernels
            logp = batched_logprobs(self.decoder, row_emb.float(), col_emb.float(), td["distance_matrix"].float(),
                                    td["duration_matrix"].float() if self.env_name == "rcvrptw" else None, inputs,
                                    out["actions"], S, temperature, tanh_clipping,
                                    autocast_dtype=self.train_replay_autocast)
            if not bool((logp > -1000).all()):
                raise AssertionError("Logprobs should not be -inf, check sampling procedure!")
            outdict["log_likelihood"] = logp.sum(1) if return_sum_log_likelihood else torch.cat(
                [torch.zeros_like(logp[:, :1]), logp], 1)
        if calc_reward and env.normalize:
            outdict["normalized_reward"] = out["normalized_reward"]
        if return_actions:
            outdict["actions"] = out["actions"]
        if select_best and S > 1:
            outdict = select_best_rows(outdict, S)
        if return_hidden:
            outdict["hidden"] = cache
        return outdict


FALLBACKS = {"softmax_range": 0}  # rollouts re-run through the per-step pipeline (diagnostics)


def filter_args(top_k=None, top_p=None) -> Tuple[int, float]:
    """rl4co's `top_k` / `top_p` decoding arguments as (int, float), None meaning off; raises ValueError for values the
    kernels reject (top_k < 0, top_p outside [0, 1] or NaN), before anything is launched."""
    k = 0 if top_k is None else top_k
    p = 0.0 if top_p is None else top_p
    if isinstance(k, bool) or int(k) != k or k < 0:
        raise ValueError(f"top_k must be a non-negative integer (got {top_k!r})")
    p = float(p)
    if not 0.0 <= p <= 1.0:  # (NaN fails too)
        raise ValueError(f"top_p must be in [0, 1] (got {top_p!r})")
    return int(k), p


def filter_active(top_k: int, top_p: float) -> bool:
    """True when the filters can drop an entry (top_k > 0, or 0 < top_p < 1)."""
    return top_k > 0 or 0.0 < top_p < 1.0


def beam_args(beam_width) -> int:
    """rl4co's `beam_width` as an int; ValueError below 2 (BeamSearch asserts beam_width > 1), NotImplementedError above
    what rrnco_beam_select serves; both before anything is launched."""
    if isinstance(beam_width, bool) or int(beam_width) != beam_width or beam_width < 2:
        raise ValueError(f"beam width must be an integer >= 2 (got {beam_width!r})")
    if beam_width > _lib.MAX_BEAM_WIDTH:
        raise NotImplementedError(f"beam width above {_lib.MAX_BEAM_WIDTH} (got {beam_width})")
    return int(beam_width)


def select_best_rows(outdict: dict, num_starts: int) -> dict:
    """rl4co's _select_best on the [num_starts * B] outputs in (s b) order: per instance the row of highest reward, the
    lowest s among equal rewards; every [num_starts * B]-leading tensor of `outdict` is cut to those B rows."""
    reward = outdict["reward"]
    R = reward.shape[0]
    B = R // num_starts
    rows = reward.view(num_starts, B).argmax(0) * B + torch.arange(B, device=reward.device)
    return {k: (v[rows] if isinstance(v, Tensor) and v.dim() >= 1 and v.shape[0] == R else v) for k, v in outdict.items()}


class SoftmaxRangeError(RuntimeError):
    """RRNCO_DEV_SOFTMAX_RANGE: the key-tiled fused kernel cannot represent this model's attention scores; its outputs
    were discarded (use stepwise_rollout)."""


_WS_CACHE = {}


def _workspace(dev, nbytes: int):
    """Scratch for rrnco_rollout, kept per (device, stream) across calls (grown when a larger batch arrives): kernels on
    one stream are ordered, so consecutive rollouts can share it."""
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), torch.cuda.current_stream(dev).cuda_stream)
    ws = _WS_CACHE.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _WS_CACHE[key] = ws
    return ws


def fused_rollout(decoder: RRNetDecoder, cache: PrecomputedCache, env, td, num_starts: int, multistart: bool,
                  kind: str, forced_actions=None, seed: int = 0, temperature: float = 1.0, tanh_clipping: float = 10.0,
                  calc_reward: bool = True, per_step_logprobs: bool = False, check: bool = True,
                  t_cap: Optional[int] = None, top_k: int = 0, top_p: float = 0.0) -> dict:
    """policy.py:203-243 as ONE kernel launch (+ a finalize kernel).  `td` is the reset td ([n_inst] batch).
    top_k / top_p: rl4co's logit filters (N <= 128 only; larger N: stepwise_rollout)."""
    top_k, top_p = filter_args(top_k, top_p)
    name = decoder.env_name
    dev = cache.glimpse_key.device
    n_inst, N, _ = cache.glimpse_key.shape
    S = int(num_starts)
    R = n_inst * S
    if N > _lib.MAX_NODES_FUSED:
        raise NotImplementedError(f"fused rollout supports N <= {_lib.MAX_NODES_FUSED} nodes (got {N})")
    if filter_active(top_k, top_p) and N > _lib.MAX_NODES_TILE:
        raise NotImplementedError(f"top_k / top_p in the fused rollout need N <= {_lib.MAX_NODES_TILE} (got {N}): use "
                                  "stepwise_rollout")
    num_loc = getattr(getattr(env, "generator", None), "num_loc", None)
    if multistart and num_loc is not None and num_loc != (N if name == "atsp" else N - 1):
        # select_start_nodes is `arange(S) % generator.num_loc` upstream; the kernel derives it from the instance size
        raise ValueError(f"env.generator.num_loc = {num_loc} does not match the instance size ({N} nodes): the fused "
                         "kernel's start-node rule would differ from env.select_start_nodes")
    if t_cap is None:
        t_cap = N if name == "atsp" else 2 * N
    forced, forced_T = None, 0
    if kind == "evaluate":
        fa = forced_actions.to(dev).contiguous()
        forced, forced_T = fa, fa.shape[1]  # the given decisions follow the forced start (policy.py:214-218)
        t_cap = max(t_cap, forced_T + (1 if multistart else 0))
    has_minmax = "min_distance" in td.keys()
    ws_bytes = _lib.lib().rrnco_rollout_workspace_bytes(ENV_ID[name], N, n_inst, S)
    ws = _workspace(dev, ws_bytes)
    seed = int(seed) & (2**63 - 1)
    from . import torch_ops
    if torch_ops.enabled():
        # dispatcher op over the same C entry point (csrc/torch_ops.cpp); outputs come from the caching allocator
        wt, alpha, beta = decoder.kernel_weight_tensors()
        acts, logp, ll, norm, real, info, _ = torch_ops.ops().rollout(
            ENV_ID[name], S, bool(multistart), DECODE_ID[kind], seed, wt, alpha, beta, float(tanh_clipping), float(temperature),
            [cache.glimpse_key, cache.glimpse_val, cache.logit_key, cache.ctx_node_proj, cache.ctx_node_proj2],
            instance_tensors_from_td(name, td), forced, t_cap, bool(per_step_logprobs), ws, top_k, top_p)
        _lib.count_call("rrnco_rollout")
        real = real if has_minmax else None
    else:
        keep = []
        w, keep_w = decoder.kernel_weights(temperature, tanh_clipping)
        data = instance_data_from_td(name, td, keep)
        acts = torch.empty((R, t_cap), dtype=torch.int64, device=dev)
        logp = torch.empty((R, t_cap), dtype=torch.float32, device=dev) if per_step_logprobs else None
        ll = torch.empty(R, dtype=torch.float32, device=dev)
        norm = torch.empty(R, dtype=torch.float32, device=dev)
        real = torch.empty(R, dtype=torch.float32, device=dev) if has_minmax else None
        info = torch.zeros(2, dtype=torch.int32, device=dev)  # [max_steps, status]
        cs = cache.struct()
        call("rrnco_rollout_filtered", ENV_ID[name], N, n_inst, S, int(multistart), DECODE_ID[kind], seed,
             C.byref(w), C.byref(cs), C.byref(data), ptr(forced), forced_T, t_cap, ptr(acts), ptr(logp), ptr(ll),
             ptr(norm), ptr(real), ptr(info[0:1]), ptr(info[1:2]), ptr(ws), min(top_k, 2**31 - 1), top_p, stream_ptr(dev))
    T, status = info.tolist()  # the ONE host sync of the rollout (upstream: 3-5 per decode step)
    if status & _lib.DEV_SOFTMAX_RANGE:  # never silently inaccurate, whatever `check` says
        raise SoftmaxRangeError("attention scores outside the range of the key-tiled kernel's fixed softmax shift")
    if check:
        _lib.raise_device_status(status)
    out = {"actions": acts[:, :T], "log_likelihood": ll}
    # decode steps each (instance, start tile) CTA actually ran (it stops when ITS rollouts are done): what the
    # roofline accounting of bench.py counts, instead of the global maximum T
    tile_rows = _lib.lib().rrnco_rollout_tile_rows(ENV_ID[name], N, n_inst, S)
    n_tiles = n_inst * ((S + tile_rows - 1) // tile_rows)
    out["tile_steps"] = ws[2 * R * 8: 2 * R * 8 + 4 * n_tiles].view(torch.int32)
    if per_step_logprobs:
        out["logprobs"] = logp[:, :T]
    if calc_reward:
        if env.normalize and has_minmax:
            out["reward"], out["normalized_reward"] = real, norm
        else:
            out["reward"] = norm
    else:  # upstream returns the (all-zero) step reward of the last env.step
        out["reward"] = torch.zeros(R, dtype=torch.float32 if name == "rcvrptw" else torch.bool, device=dev)
    return out


def select_action(logits, mask, kind: str = "greedy", tanh_clipping: float = 10.0, temperature: float = 1.0,
                  seed: int = 0, step: int = 0, forced_action=None, status=None, top_k: int = 0, top_p: float = 0.0):
    """DecodingStrategy.step (decoding.py:219-298): (action int64 [R], log-prob fp32 [R]) in one kernel, with rl4co's
    top_k / top_p logit filters (decoding.py:311-361; include/rrnco_b200.h describes the tie rule)."""
    top_k, top_p = filter_args(top_k, top_p)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=logits.device)
    from . import torch_ops
    if torch_ops.enabled():
        _lib.count_call("rrnco_select_action")
        action, logp = torch_ops.ops().select_action(logits, mask, DECODE_ID[kind], float(tanh_clipping), float(temperature),
                                                     int(seed) & (2**63 - 1), int(step), forced_action, status, top_k,
                                                     top_p)
        return action, logp, status
    logits, mask = logits.contiguous(), mask.contiguous()
    R, N = logits.shape
    action = torch.empty(R, dtype=torch.int64, device=logits.device)
    logp = torch.empty(R, dtype=torch.float32, device=logits.device)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=logits.device)
    forced = None if forced_action is None else forced_action.contiguous()
    call("rrnco_select_action_filtered", R, N, ptr(logits), ptr(_u8(mask)), DECODE_ID[kind], float(tanh_clipping),
         float(temperature), int(seed) & (2**63 - 1), int(step), ptr(forced), ptr(action), ptr(logp), ptr(status),
         min(top_k, 2**31 - 1), top_p, stream_ptr(logits.device))
    return action, logp, status


_ROLLOUT_STATE_KEYS = {
    "atsp": ("first_node", "current_node", "i", "action_mask"),
    "rcvrp": ("current_node", "used_capacity", "vehicle_capacity", "visited", "action_mask"),
    "rcvrptw": ("current_node", "current_time", "current_route_length", "used_capacity_linehaul",
                "used_capacity_backhaul", "visited", "action_mask", "vehicle_capacity", "open_route", "distance_limit",
                "backhaul_class"),
}


def stepwise_rollout(decoder: RRNetDecoder, cache: PrecomputedCache, env, td, num_starts: int, multistart: bool,
                     kind: str, forced_actions=None, seed: int = 0, temperature: float = 1.0, tanh_clipping: float = 10.0,
                     calc_reward: bool = True, per_step_logprobs: bool = False, check: bool = True, t_cap=None,
                     top_k: int = 0, top_p: float = 0.0) -> dict:
    """policy.py:203-243 as a per-step kernel pipeline for ANY number of nodes (decoder_logits_large ->
    select_action -> env step), used when N exceeds the fused kernel's 128-key tile.  Only the rollout STATE is
    replicated over the POMO starts; matrices / demands / time windows stay one copy per instance (the kernels
    index row r % data_rows), so the n=1000 configs never materialise upstream's S-fold `batchify` of [N,N] data.
    top_k / top_p: rl4co's logit filters, for any N."""
    top_k, top_p = filter_args(top_k, top_p)
    from .tdlite import TensorDictLite, batchify
    from .envs import tour_reward
    name = decoder.env_name
    n_inst, N, _ = cache.glimpse_key.shape
    S = int(num_starts)
    R = n_inst * S
    dev = cache.glimpse_key.device
    roll = {k: (batchify(td[k], S) if k in _ROLLOUT_STATE_KEYS[name] else td[k]) for k in td.keys() if k != "done"}
    roll = TensorDictLite(roll, batch_size=[R])
    actions, logps = [], []
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    if multistart:
        a0 = env.select_start_nodes(td, S)
        roll.set("action", a0)
        roll = env.step(roll)["next"]
        actions.append(a0)
        logps.append(torch.zeros(R, dtype=torch.float32, device=dev))
        done = roll["done"]
    else:
        done = torch.zeros(R, dtype=torch.bool, device=dev)
    step = 0
    max_steps = 2 * N + 2
    while step < max_steps:
        if name == "atsp":  # fixed length: no host sync needed
            if len(actions) >= N:
                break
        elif bool(done.all()):  # upstream syncs here every step too (policy.py:212)
            break
        logits, mask = decoder(roll, cache, S)
        forced = forced_actions[:, step].to(dev) if kind == "evaluate" else None
        a, lp, status = select_action(logits, mask, kind, tanh_clipping, temperature, seed, step, forced, status, top_k, top_p)
        roll.set("action", a)
        roll = env.step(roll)["next"]
        done = roll["done"]
        actions.append(a)
        logps.append(lp)
        step += 1
    if check:
        _lib.raise_device_status(int(status.item()))
    acts = torch.stack(actions, 1)
    lps = torch.stack(logps, 1)
    out = {"actions": acts, "log_likelihood": lps.double().sum(1).float(), "logprobs": lps}
    has_minmax = "min_distance" in td.keys()
    if calc_reward:
        open_route = td["open_route"] if name == "rcvrptw" else None
        real, norm = tour_reward(acts, td["distance_matrix"], name != "atsp", open_route,
                                 td["min_distance"] if has_minmax and env.normalize else None,
                                 td["max_distance"] if has_minmax and env.normalize else None)
        if env.normalize and has_minmax:
            out["reward"], out["normalized_reward"] = real, norm
        else:
            out["reward"] = norm
    else:
        out["reward"] = torch.zeros(R, dtype=torch.float32 if name == "rcvrptw" else torch.bool, device=dev)
    return out


def beam_select(logits, mask, score, beam_width: int, tanh_clipping: float = 10.0, temperature: float = 1.0, status=None):
    """One BeamSearch step (rl4co decoding.py:402-542, _make_beam_step) over the [W * B, N] decoder output in (w b) order:
    (action int64, parent row int64, log-prob fp32, new score fp32), each [W * B].  Candidates are ranked by (value
    descending, flat index w * N + n ascending); include/rrnco_b200.h (rrnco_beam_select) gives the full rule."""
    W = beam_args(beam_width)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=logits.device)
    from . import torch_ops
    if torch_ops.enabled():
        _lib.count_call("rrnco_beam_select")
        action, parent, logp, new_score = torch_ops.ops().beam_select(logits, mask, score, W, float(tanh_clipping),
                                                                      float(temperature), status)
        return action, parent, logp, new_score, status
    logits, mask, score = logits.float().contiguous(), mask.contiguous(), score.float().contiguous()
    R, N = logits.shape
    if R % W:
        raise ValueError(f"{R} rows are not a whole number of beams of width {W}")
    action = torch.empty(R, dtype=torch.int64, device=logits.device)
    parent = torch.empty(R, dtype=torch.int64, device=logits.device)
    logp = torch.empty(R, dtype=torch.float32, device=logits.device)
    new_score = torch.empty(R, dtype=torch.float32, device=logits.device)
    call("rrnco_beam_select", R // W, W, N, ptr(logits), ptr(_u8(mask)), ptr(score), float(tanh_clipping),
         float(temperature), ptr(action), ptr(parent), ptr(logp), ptr(new_score), ptr(status), stream_ptr(logits.device))
    return action, parent, logp, new_score, status


def beam_backtrack(actions, parents, logprobs, per_step_logprobs: bool = True, status=None):
    """BeamSearch._backtrack: step-major [T, R] actions / parent rows / log-probs -> (actions [R, T], aligned log-probs
    [R, T] or None, log-likelihood [R], status).  A parent row outside [0, R) sets DEV_BAD_PARENT in `status`."""
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=actions.device)
    from . import torch_ops
    if torch_ops.enabled():
        _lib.count_call("rrnco_beam_backtrack")
        a, lp, ll = torch_ops.ops().beam_backtrack(actions, parents, logprobs, bool(per_step_logprobs), status)
        return a, (lp if per_step_logprobs else None), ll, status
    actions, parents, logprobs = actions.contiguous(), parents.contiguous(), logprobs.float().contiguous()
    T, R = actions.shape
    dev = actions.device
    a = torch.empty((R, T), dtype=torch.int64, device=dev)
    lp = torch.empty((R, T), dtype=torch.float32, device=dev) if per_step_logprobs else None
    ll = torch.empty(R, dtype=torch.float32, device=dev)
    call("rrnco_beam_backtrack", R, T, ptr(actions), ptr(parents), ptr(logprobs), ptr(a), ptr(lp), ptr(ll), ptr(status),
         stream_ptr(dev))
    return a, lp, ll, status


def fused_beam_serves(env_name: str, n_nodes: int, beam_width: int) -> bool:
    """Whether rrnco_beam_rollout serves a beam search of this size: N <= 112 and 2..128 beams, under the default engine and
    precision (rrnco_set_ffn_engine(2), rrnco_set_precision(3)); beam_search_rollout serves every other call."""
    return _lib.lib().rrnco_beam_rollout_workspace_bytes(ENV_ID[env_name], int(n_nodes), 1, int(beam_width)) > 0


def fused_beam_rollout(decoder: RRNetDecoder, cache: PrecomputedCache, env, td, beam_width: int,
                       temperature: float = 1.0, tanh_clipping: float = 10.0, calc_reward: bool = True,
                       per_step_logprobs: bool = False, check: bool = True) -> dict:
    """beam_search_rollout in one launch of the lean rollout kernel (rrnco_beam_rollout): one CTA per instance whose W rows
    are the beams; same rule, same outputs.  N <= 112 and W <= 128 under the default engine and precision only
    (fused_beam_serves); NotImplementedError otherwise."""
    W = beam_args(beam_width)
    name = decoder.env_name
    dev = cache.glimpse_key.device
    n_inst, N, _ = cache.glimpse_key.shape
    R = n_inst * W
    ws_bytes = _lib.lib().rrnco_beam_rollout_workspace_bytes(ENV_ID[name], N, n_inst, W)
    if ws_bytes <= 0:
        raise NotImplementedError(f"the fused beam search serves N <= {_lib.MAX_NODES_LEAN} and beam widths up to "
                                  f"{_lib.MAX_BEAM_WIDTH_FUSED} under the default engine and precision (got N={N}, W={W}): "
                                  "use beam_search_rollout")
    num_loc = getattr(getattr(env, "generator", None), "num_loc", None)
    if num_loc is not None and num_loc != (N if name == "atsp" else N - 1):
        raise ValueError(f"env.generator.num_loc = {num_loc} does not match the instance size ({N} nodes): the fused "
                         "kernel's start-node rule would differ from env.select_start_nodes")
    t_cap = N if name == "atsp" else 2 * N + 3  # the per-step loop's bound (beam_search_rollout)
    ws = _workspace(dev, ws_bytes)
    from . import torch_ops
    if torch_ops.enabled():
        wt, alpha, beta = decoder.kernel_weight_tensors()
        acts, parents, lps, info = torch_ops.ops().beam_rollout(
            ENV_ID[name], W, wt, alpha, beta, float(tanh_clipping), float(temperature),
            [cache.glimpse_key, cache.glimpse_val, cache.logit_key, cache.ctx_node_proj, cache.ctx_node_proj2],
            instance_tensors_from_td(name, td), t_cap, ws)
        _lib.count_call("rrnco_beam_rollout")
    else:
        keep = []
        w, keep_w = decoder.kernel_weights(temperature, tanh_clipping)
        data = instance_data_from_td(name, td, keep)
        acts = torch.empty((t_cap, R), dtype=torch.int64, device=dev)
        parents = torch.empty((t_cap, R), dtype=torch.int64, device=dev)
        lps = torch.empty((t_cap, R), dtype=torch.float32, device=dev)
        info = torch.zeros(2, dtype=torch.int32, device=dev)  # [steps, status]
        cs = cache.struct()
        call("rrnco_beam_rollout", ENV_ID[name], N, n_inst, W, C.byref(w), C.byref(cs), C.byref(data), t_cap, ptr(acts),
             ptr(parents), ptr(lps), ptr(info[0:1]), ptr(info[1:2]), ptr(ws), stream_ptr(dev))
    T = int(info[0].item())
    acts, lps, ll, status = beam_backtrack(acts[:T], parents[:T], lps[:T], per_step_logprobs, info[1:2])
    if check:
        _lib.raise_device_status(int(status.item()))
    return _beam_outputs(name, env, td, acts, lps, ll, per_step_logprobs, calc_reward)


def _beam_outputs(name, env, td, acts, lps, ll, per_step_logprobs, calc_reward) -> dict:
    """The out-dict of a beam search from its backtracked sequences: actions, log_likelihood, logprobs, rewards."""
    out = {"actions": acts, "log_likelihood": ll}
    if per_step_logprobs:
        out["logprobs"] = lps
    has_minmax = "min_distance" in td.keys()
    if calc_reward:
        open_route = td["open_route"] if name == "rcvrptw" else None
        real, norm = tour_reward(acts, td["distance_matrix"], name != "atsp", open_route,
                                 td["min_distance"] if has_minmax and env.normalize else None,
                                 td["max_distance"] if has_minmax and env.normalize else None)
        if env.normalize and has_minmax:
            out["reward"], out["normalized_reward"] = real, norm
        else:
            out["reward"] = norm
    else:
        out["reward"] = torch.zeros(acts.shape[0], dtype=torch.float32 if name == "rcvrptw" else torch.bool,
                                    device=acts.device)
    return out


def beam_search_rollout(decoder: RRNetDecoder, cache: PrecomputedCache, env, td, beam_width: int,
                        temperature: float = 1.0, tanh_clipping: float = 10.0, calc_reward: bool = True,
                        per_step_logprobs: bool = False, check: bool = True) -> dict:
    """rl4co BeamSearch (decoding.py:402-542) as a per-step kernel pipeline for any N: decoder_logits -> beam_select ->
    the rollout state of each new beam gathered from its parent row -> env step, then beam_backtrack.  Rows r = w * B + b;
    the start nodes are env.select_start_nodes(td, W) with log-prob 0.  Only the rollout state is replicated over the
    beams (what stepwise_rollout replicates), never the instance matrices.  Returns the [W * B] outputs of every beam."""
    W = beam_args(beam_width)
    from .tdlite import TensorDictLite, batchify
    name = decoder.env_name
    n_inst, N, _ = cache.glimpse_key.shape
    R = n_inst * W
    dev = cache.glimpse_key.device
    state_keys = _ROLLOUT_STATE_KEYS[name]
    roll = {k: (batchify(td[k], W) if k in state_keys else td[k]) for k in td.keys() if k != "done"}
    roll = TensorDictLite(roll, batch_size=[R])
    a0 = env.select_start_nodes(td, W)
    roll.set("action", a0)
    roll = env.step(roll)["next"]
    actions, parents, logps = [a0], [torch.zeros(R, dtype=torch.int64, device=dev)], [torch.zeros(R, device=dev)]
    score = torch.zeros(R, dtype=torch.float32, device=dev)
    done = roll["done"]
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    max_steps = 2 * N + 2
    while len(actions) <= max_steps:
        if name == "atsp":  # fixed length: no host sync needed
            if len(actions) >= N:
                break
        elif bool(done.all()):
            break
        logits, mask = decoder(roll, cache, W)
        a, parent, lp, score, status = beam_select(logits, mask, score, W, tanh_clipping, temperature, status)
        for k in state_keys:  # each new beam continues from its parent's state
            roll[k] = roll[k].index_select(0, parent)
        roll.set("action", a)
        roll = env.step(roll)["next"]
        done = roll["done"]
        actions.append(a)
        parents.append(parent)
        logps.append(lp)
    acts, lps, ll, status = beam_backtrack(torch.stack(actions), torch.stack(parents), torch.stack(logps),
                                           per_step_logprobs, status)
    if check:
        _lib.raise_device_status(int(status.item()))
    return _beam_outputs(name, env, td, acts, lps, ll, per_step_logprobs, calc_reward)
