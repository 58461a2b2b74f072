"""B200-native embedding + FM / cross hot path of the reference's Deep-CTR models.

The directory name carries a hyphen (it mirrors the reference's name); import it with
`importlib.import_module("details-in-recommendation_b200")` or through the alias module
`dir_b200` at the repository root.
"""
from . import _lib, roofline, synth                          # noqa: F401
from ._lib import LIB_PATH, build, launch_count             # noqa: F401
from .bags import EmbeddingBagFM                              # noqa: F401
from .feeder import ColumnFeeder, HostFeeder                              # noqa: F401
from . import frontend                                         # noqa: F401
from .frontend import FeatureFrontEnd                          # noqa: F401
from .layers import CrossNetwork, EmbeddingFM, InputLayer, SortedLookups # noqa: F401
from .models import DCN, DeepFM, TFAdam                       # noqa: F401
from .sharded import ShardedEmbeddingBagFM, ShardedEmbeddingFM, ShardedLookups, ShardPlan  # noqa: F401

__all__ = ["DeepFM", "DCN", "TFAdam", "EmbeddingFM", "EmbeddingBagFM", "InputLayer", "CrossNetwork", "ShardedEmbeddingFM", "ShardedEmbeddingBagFM", "ShardPlan", "HostFeeder", "ColumnFeeder", "FeatureFrontEnd", "frontend", "synth", "roofline", "build", "launch_count", "LIB_PATH"]
