"""lightzero_b200 -- B200-native batched MuZero MCTS + model inference behind the reference's own
interfaces (lzero.mcts.tree_search.MuZeroMCTSCtree, lzero.mcts.ctree.ctree_muzero.mz_tree,
lzero.model.MuZeroModel; plus the EfficientZero counterparts EfficientZeroMCTSCtree, ez_tree, EfficientZeroModel, and the Gumbel MuZero search GumbelMuZeroMCTSCtree, gmz_tree).  All compute is hand-written sm_100a CUDA behind the C ABI of
include/lzb200.h; this package is the thin host side."""
from .mcts_ctree import EfficientZeroMCTSCtree, GumbelMuZeroMCTSCtree, MuZeroMCTSCtree, UniZeroMCTSCtree  # noqa: F401
from .efficientzero_model import EfficientZeroModel, EZNetworkOutput  # noqa: F401
from .muzero_model import MuZeroModel, MZNetworkOutput  # noqa: F401
from .muzero_model_mlp import MuZeroModelMLP  # noqa: F401
from .scaling_transform import DiscreteSupport, InverseScalarTransform  # noqa: F401
from . import ez_tree, gmz_tree, mz_tree  # noqa: F401

__all__ = ["MuZeroMCTSCtree", "EfficientZeroMCTSCtree", "GumbelMuZeroMCTSCtree", "gmz_tree", "UniZeroMCTSCtree", "EfficientZeroModel", "EZNetworkOutput", "ez_tree", "MuZeroModel", "MuZeroModelMLP", "MZNetworkOutput", "DiscreteSupport",
           "InverseScalarTransform", "mz_tree"]
