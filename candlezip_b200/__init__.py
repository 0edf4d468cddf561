"""candlezip_b200: B200-native (sm_100a) implementation of CandleZip's model-driven entropy-coding hot path,
behind the reference's LanguageModelSession boundary.  See DESIGN.md and include/candlezip_b200.h."""
from ._lib import (CZ_ARCH_RWKV7, CZ_ARCH_SMOLLM, CZ_CDF_RWKV_LITERALS, CZ_CDF_SMOLLM, CZ_CDF_SMOLLM_FLOOR,  # noqa: F401
                   CZ_ENGINE_SIMT, CZ_ENGINE_TCGEN05, CzError)
from .api import RWKV7_0P1B, SMOLLM_135M, SMOLLM_TINY, Context, Model, Session, split_segments, xe_make_prime  # noqa: F401
from . import codec, container, gate, sharding  # noqa: F401
