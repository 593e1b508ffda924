"""rrnco_b200 -- B200-native (sm_100a) construction-rollout hot path of ai4co/real-routing-nco.

Host-side mirror of the reference interface for this path (same class / method names, td schema and error
texts) on top of the C-ABI library `librrnco_b200.so` (include/rrnco_b200.h):

    from rrnco_b200 import ATSPEnv, RCVRPEnv, RMTVRPEnv            # rrnco.envs.{atsp,rcvrp,rmtvrp}
    from rrnco_b200 import RRNetDecoder, RRNetPolicy              # rrnco.models
    from rrnco_b200 import Real_World_Sampler                     # rrnco.envs.*.sampler

No CPU fallback, no Triton / torch.compile: if the CUDA library is missing, calls raise.
"""
from ._lib import RRNCOError, set_ffn_engine, set_precision, set_step_tiling  # noqa: F401
from .envs import ATSPEnv, RCVRPEnv, RMTVRPEnv, get_env  # noqa: F401
from .models import (PrecomputedCache, RRNetDecoder, RRNetPolicy, beam_backtrack, beam_search_rollout,  # noqa: F401
                     beam_select, fused_rollout, select_action, stepwise_rollout)
from .dataio import iter_batches, load_city_npz, load_npz_to_tensordict, prepare_test_td  # noqa: F401
from .hostio import HostPrefetcher  # noqa: F401
from .sampler import CityOnDevice, Real_World_Sampler, remove_outlier_points  # noqa: F401
from .generator import LazyATSPGenerator, LazyRCVRPGenerator, LazyRMTVRPGenerator  # noqa: F401
from .transforms import StateAugmentation, dihedral_8_augmentation  # noqa: F401
from .tdlite import TensorDictLite, batchify, unbatchify  # noqa: F401
from .torch_ops import use_torch_ops  # noqa: F401
from .encoder_ops import DistAngleFusion, aft_nab, patch_encoder  # noqa: F401
from .training import (batched_logprobs, collect_decode_inputs, iter_decode_inputs, pomo_shared_baseline_loss,  # noqa: F401
                       replay_log_likelihood)

__all__ = ["ATSPEnv", "RCVRPEnv", "RMTVRPEnv", "get_env", "RRNetDecoder", "RRNetPolicy", "PrecomputedCache",
           "fused_rollout", "stepwise_rollout", "select_action", "beam_search_rollout", "beam_select", "beam_backtrack", "Real_World_Sampler", "TensorDictLite", "batchify", "unbatchify", "set_precision", "set_ffn_engine", "set_step_tiling",
           "RRNCOError", "HostPrefetcher", "load_city_npz", "load_npz_to_tensordict", "prepare_test_td", "iter_batches", "replay_log_likelihood", "batched_logprobs", "collect_decode_inputs", "iter_decode_inputs",
           "pomo_shared_baseline_loss", "CityOnDevice", "remove_outlier_points", "LazyATSPGenerator", "LazyRCVRPGenerator",
           "LazyRMTVRPGenerator", "StateAugmentation", "dihedral_8_augmentation"]
