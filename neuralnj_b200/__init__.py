"""neuralnj_b200 — B200-native (sm_100a) inference hot path of NeuralNJ behind the reference's Python API.

    from neuralnj_b200 import PhyloATTN, PhyInferEnv, reinforce_rollout, Argmax_inference, load_pi_instance

CUDA kernels live in csrc/ and are reached through the C ABI of include/nnj.h (libnnj.so).
"""
from ._lib import NnjError, build, lib            # noqa: F401
from .config import CfgNode, empty_config, inference_config   # noqa: F401
from .environment import PhyInferEnv, PhyloTree, format_rtree   # noqa: F401
from .model import PhyloATTN                        # noqa: F401
from .phydata import load_pi_instance               # noqa: F401
from .rollout import (Agmax_one_instance, Argmax_inference, RL_Search, Search_inference,   # noqa: F401
                      reinforce_rollout)
from .treeutil import rf_distance, treestr_to_tuples   # noqa: F401
from .likelihood import compute_llh, optimize_brlen          # noqa: F401
from .supervise import balanced_elu_loss, supervise_rollout   # noqa: F401
from .support import bootstrap_support, likelihood_support, topology_test        # noqa: F401

__all__ = ["PhyloATTN", "PhyInferEnv", "PhyloTree", "reinforce_rollout", "Agmax_one_instance", "Argmax_inference",
           "RL_Search", "Search_inference", "load_pi_instance", "empty_config", "inference_config", "CfgNode",
           "rf_distance", "treestr_to_tuples", "format_rtree", "build", "lib", "NnjError", "optimize_brlen", "compute_llh",
           "supervise_rollout", "balanced_elu_loss", "bootstrap_support", "likelihood_support",
           "topology_test"]
