"""mil_b200 — B200-native (sm_100a) implementation of the multimodal MIL aggregator hot path of
KyleKWKim/LLM-guided-Multimodal-MIL behind the reference's nn.Module interfaces.

The directory name carries hyphens, so import it through the repo-root shim: ``import mil_b200``.
"""
from . import _lib
from ._lib import MilB200Error, launch_count, lib
from . import functional
from .abmil import ABMIL, ABMIL_v2
from . import model
from . import clip_loss
from . import feeder
from .feeder import PackedBagFeeder, ResidentBagFeeder, pack_bags_host
from .fusion_trainer import FusionTrainer
from .clip_loss import CLIPLogits, CLIPloss_v1
from .model.sam.transformer import Attention, TwoWayAttentionBlock, TwoWayTransformer
from .model.sam.common import MLPBlock
from .model.utils import get_model

__all__ = ["ABMIL", "ABMIL_v2", "Attention", "TwoWayAttentionBlock", "TwoWayTransformer", "MLPBlock", "CLIPLogits",
           "CLIPloss_v1", "get_model", "model", "clip_loss", "functional", "lib", "launch_count", "MilB200Error"]
