"""B200-native drop-in for the reference bridge hot path.

Reference: src/vlm_bridge/model_architecture/bridge_module.py (BridgeLite and its blocks).
"""
__version__ = "0.1.0"

from .bridge import (BridgeBlock, BridgeLite, MultiHeadCrossAttention,  # noqa: E402,F401
                     MultiHeadSelfAttention)
from . import checkpoint  # noqa: E402,F401
from .decode import DecodeStepGraphs, beam_search_decode, greedy_decode  # noqa: E402,F401
from .graph import GraphedBridgeStep  # noqa: E402,F401
from .kv_cache import VisionKVCache  # noqa: E402,F401
from .loss import FusedCrossEntropyLoss, fused_cross_entropy  # noqa: E402,F401
from .optim import BridgeAdamW  # noqa: E402,F401
