"""B200-native batched implementation of the RIS-VEC `Environ.step/reset` hot path.

`BatchedEnviron` (batched.py) is the host-side mirror of the reference class; it drives
hand-written sm_100a kernels through the C ABI in include/risvec.h.  The CUDA library is
mandatory: importing `BatchedEnviron` works without a GPU, constructing one does not.
"""
from ._lib import (EP_STAGES, PARTNER_NONE, PARTNER_SECOND, PARTNER_SINGLE, STAT_COLUMNS, RisvecError,
                   RisvecLibraryError, build_library, load_library)
from .batched import (MARL_TRACES, SARL_TRACES, BatchedEnviron, default_pairing, default_params, encode_groups,
                      marl_yaml_overrides, mask_schedule)
from .episode_log import EpisodeLog
from .replay import ReplayBuffer

__all__ = ["BatchedEnviron", "EpisodeLog", "ReplayBuffer", "default_params", "default_pairing", "mask_schedule",
           "encode_groups", "marl_yaml_overrides", "build_library",
           "load_library", "RisvecError", "RisvecLibraryError", "MARL_TRACES", "SARL_TRACES", "STAT_COLUMNS",
           "PARTNER_NONE", "PARTNER_SECOND", "PARTNER_SINGLE", "EP_STAGES"]
