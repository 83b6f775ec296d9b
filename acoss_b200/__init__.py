"""acoss_b200 — B200-native (sm_100a) implementation of acoss's all-pairs cover-song scoring
hot path (OTI -> HPCP cross-similarity -> binary CRP -> Qmax / Smith-Waterman), behind the
reference's CoverAlgorithm plugin API.  See DESIGN.md."""
from ._lib import AcossError, Params, default_params  # noqa: F401
from .engine import Engine, pack_tracks  # noqa: F401
from .simple import Simple  # noqa: F401

__version__ = "0.1.0"
