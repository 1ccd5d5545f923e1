"""Device-resident mirror of the reference's Cython module ``lzero.mcts.ctree.ctree_gumbel_muzero.gmz_tree``
(gmz_tree.pyx:5-152): ``Roots``, ``MinMaxStatsList``, ``ResultsWrapper``, ``batch_traverse``, ``batch_back_propagate`` with the
reference's names and argument order.  The trees are the CUDA trees of ``mz_tree`` switched to Gumbel mode
(``lz_tree_set_gumbel``, csrc/gumbel.cu): root choice by sequential halving over a fixed Gumbel draw, interior choice by the
completed-Q improved policy.  Nothing on the search path is random, so the results are the reference's bit for bit.

As in ``mz_tree``, every list argument may also be a numpy array or a CUDA tensor, list results cost one device->host copy and
``*_tensor`` variants stay on the device.  ``MinMaxStatsList`` is bookkeeping only: no Gumbel routine reads MinMax statistics.
"""
from typing import List

import numpy as np
import torch

from . import cabi
from .mz_tree import DEFAULT_MAX_SIMS, MinMaxStatsList, ResultsWrapper, TreeHandle, _to_dev
from .mz_tree import Roots as _MzRoots

__all__ = ["Roots", "MinMaxStatsList", "ResultsWrapper", "batch_traverse", "batch_back_propagate"]


class Roots(_MzRoots):
    """gmz_tree.pyx:28-65.  ``legal_actions_list``: list of lists (any order), or a uint8/bool mask [root_num, A]."""

    def __init__(self, root_num: int, legal_actions_list, device=None):
        super().__init__(root_num, legal_actions_list, device)
        self._values = None
        self._gumbel = None        # (num_simulations, max_num_considered_actions) the tree is set up for

    # ---- reference API ---------------------------------------------------------------------------
    def prepare(self, root_noise_weight: float, noises, value_prefix_pool, value_pool, policy_logits_pool, to_play_batch):
        self._values = _to_dev(value_pool, torch.float32, self.device, (self.root_num,))
        self._stage(float(root_noise_weight), noises, value_prefix_pool, policy_logits_pool, to_play_batch)

    def prepare_no_noise(self, value_prefix_pool, value_pool, policy_logits_pool, to_play_batch):
        self._values = _to_dev(value_pool, torch.float32, self.device, (self.root_num,))
        self._stage(0.0, None, value_prefix_pool, policy_logits_pool, to_play_batch)

    def get_children_values(self, discount: float, action_space_size: int) -> List[List[float]]:
        return self.get_children_values_tensor(discount, action_space_size).cpu().tolist()

    def get_policies(self, discount: float, action_space_size: int) -> List[List[float]]:
        return self.get_policies_tensor(discount, action_space_size).cpu().tolist()

    # ---- device-side extras ----------------------------------------------------------------------
    def get_children_values_tensor(self, discount: float, action_space_size: int) -> torch.Tensor:
        """Completed Q values f32 [B, A] by action id, -inf for illegal actions (cnode.cpp:309-338)."""
        return self.results_tensor(discount, action_space_size)[0]

    def get_policies_tensor(self, discount: float, action_space_size: int) -> torch.Tensor:
        """Improved policy f32 [B, A] by action id, 0 for illegal actions (cnode.cpp:355-385)."""
        return self.results_tensor(discount, action_space_size)[1]

    def results_tensor(self, discount: float, action_space_size: int):
        """(children values [B,A], improved policy [B,A], arg-max action of the improved policy [B] int32), one kernel."""
        t = self._need_tree()
        assert action_space_size == t.A, f"action_space_size {action_space_size} != the roots' {t.A} actions"
        cv = torch.empty(self.root_num, t.A, device=self.device)
        pol = torch.empty(self.root_num, t.A, device=self.device)
        act = torch.empty(self.root_num, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_results_gumbel(t.h, float(discount), cv.data_ptr(), pol.data_ptr(), act.data_ptr(),
                                                    cabi.stream_ptr()), "lz_tree_results_gumbel")
        return cv, pol, act

    # ---- internals -------------------------------------------------------------------------------
    def _need_tree(self) -> TreeHandle:
        if self._tree is None:
            self._materialize(DEFAULT_MAX_SIMS, (DEFAULT_MAX_SIMS, DEFAULT_MAX_SIMS))
        return self._tree

    def _materialize(self, max_sims: int, params=None):
        """params: (num_simulations, max_num_considered_actions) of the Gumbel tables."""
        self._gumbel = tuple(params) if params is not None else (self._gumbel or (max_sims, max_sims))
        super()._materialize(max(max_sims, self._gumbel[0]))

    def _set_gumbel(self, t: TreeHandle, num_simulations: int, max_num_considered_actions: int):
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_set_gumbel(t.h, int(num_simulations), int(max_num_considered_actions)), "lz_tree_set_gumbel")
        self._gumbel = (int(num_simulations), int(max_num_considered_actions))

    def _prepare_tree(self, t: TreeHandle, p: dict, s):
        self._set_gumbel(t, *self._gumbel)
        cabi.check(t.lib.lz_tree_prepare_gumbel(t.h, p["logits"].data_ptr(), cabi.ptr(p["noise"]), p["w"], cabi.ptr(p["rewards"]),
                                                cabi.ptr(self._values), cabi.ptr(p["to_play"]), s), "lz_tree_prepare_gumbel")


def batch_traverse(roots: Roots, num_simulations: int, max_num_considered_actions: int, discount: float,
                   results: ResultsWrapper, virtual_to_play_batch, return_tensors: bool = False):
    """gmz_tree.pyx:91-95 -> (latent_state_index_in_search_path, latent_state_index_in_batch, last_actions,
    virtual_to_play_batch); the last is the argument, unchanged (cnode.cpp:894)."""
    key = (int(num_simulations), int(max_num_considered_actions))
    if roots._tree is None:
        roots._materialize(key[0], key)
    elif roots._gumbel != key:
        roots._set_gumbel(roots._tree, *key)
    t = roots._tree
    with torch.cuda.device(roots.device):
        cabi.check(t.lib.lz_tree_traverse_gumbel(t.h, float(discount), t.ix.data_ptr(), t.iy.data_ptr(), t.action.data_ptr(),
                                                 t.search_len.data_ptr(), t.vtp.data_ptr(), cabi.stream_ptr()),
                   "lz_tree_traverse_gumbel")
    results._roots = roots
    if return_tensors:
        return t.ix, t.iy, t.action, t.vtp
    packed = torch.stack((t.ix, t.iy, t.action)).cpu().numpy()
    vtp = virtual_to_play_batch.tolist() if hasattr(virtual_to_play_batch, "tolist") else list(virtual_to_play_batch)
    return packed[0].tolist(), packed[1].tolist(), packed[2].tolist(), vtp


def batch_back_propagate(current_latent_state_index: int, discount: float, value_prefixs, values, policies,
                         min_max_stats_lst: MinMaxStatsList, results: ResultsWrapper, to_play_batch):
    """gmz_tree.pyx:81-88.  ``to_play_batch`` is accepted for the reference's signature; the Gumbel back-up does not use it."""
    roots = results._roots
    t = roots._tree
    B, A = roots.root_num, t.A
    dev = roots.device
    rew = _to_dev(value_prefixs, torch.float32, dev, (B,))
    val = _to_dev(values, torch.float32, dev, (B,))
    pol = _to_dev(policies, torch.float32, dev, (B, A))
    with torch.cuda.device(dev):
        cabi.check(t.lib.lz_tree_backpropagate_gumbel(t.h, int(current_latent_state_index), float(discount), rew.data_ptr(),
                                                      val.data_ptr(), pol.data_ptr(), cabi.stream_ptr()),
                   "lz_tree_backpropagate_gumbel")
    t._keep = (rew, val, pol)
