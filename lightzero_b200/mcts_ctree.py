"""Mirror of ``lzero.mcts.tree_search.mcts_ctree.MuZeroMCTSCtree`` (mcts_ctree.py:211-368): same
class-level ``config``, ``default_config()``, ``__init__(cfg)``, ``roots(n, legal_actions)`` and
``search(roots, model, latent_state_roots, to_play_batch, task_id=None)``.

``search`` has two execution modes, both entirely on the GPU:
  * fused (``model`` is a ``lightzero_b200.MuZeroModel``): the whole num_simulations loop is one CUDA
    graph launch (``lz_search_run``) -- zero host<->device synchronisations inside the search;
  * step-wise (any other object with ``recurrent_inference``, e.g. the user's own torch module on
    CUDA): the device trees are driven one simulation at a time around the caller's model; the tree
    hands the gather indices to torch on device, so this mode also never syncs with the host.

Parity contract: ``deterministic=True`` reproduces the reference C++ ctree bit for bit (first legal
action attaining the maximum, cnode.cpp:592); the reference's default mode seeds rand() from the wall
clock on every traverse (cnode.cpp:770, utils.cpp:12-26) and is not reproducible by construction, so
``deterministic=False`` draws from the same tie list with a counter-based device RNG instead.
"""
import copy
from typing import Any, List, Optional, Union

import numpy as np
import torch

from . import cabi, ez_tree, gmz_tree, mz_tree
from .efficientzero_model import EfficientZeroModel
from .muzero_model import MuZeroModel
from .muzero_model_mlp import MuZeroModelMLP
from .scaling_transform import DiscreteSupport, InverseScalarTransform


class ConfigDict(dict):
    """Minimal attribute dict (the reference uses easydict.EasyDict, not installed here)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, ConfigDict):
            v = ConfigDict(v)
        super().__setitem__(k, v)

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v

    def update(self, other=None, **kw):
        for k, v in dict(other or {}, **kw).items():
            self[k] = v


class MuZeroMCTSCtree(object):
    # mcts_ctree.py:220-232
    config = dict(
        root_dirichlet_alpha=0.3,
        root_noise_weight=0.25,
        pb_c_base=19652,
        pb_c_init=1.25,
        value_delta_max=0.01,
        env_type='not_board_games',
    )
    # extension: tie-breaking mode (the reference MuZero search passes no flag, i.e. False)
    deterministic_default = False

    @classmethod
    def default_config(cls) -> ConfigDict:
        cfg = ConfigDict(copy.deepcopy(cls.config))
        cfg.cfg_type = cls.__name__ + 'Dict'
        return cfg

    def __init__(self, cfg=None) -> None:
        default_config = self.default_config()
        default_config.update(cfg or {})
        self._cfg = default_config
        self._cfg.setdefault("num_simulations", 50)
        self._cfg.setdefault("discount_factor", 0.997)
        self._cfg.setdefault("device", "cuda")
        self.deterministic = bool(self._cfg.get("deterministic", self.deterministic_default))
        self._inv = self._inv_reward = None    # lazily: InverseScalarTransforms for the step-wise mode (mcts_ctree.py:249-253)

    @classmethod
    def roots(cls, active_collect_env_num: int, legal_actions: List[Any]) -> "mz_tree.Roots":
        """mcts_ctree.py:255-265"""
        return mz_tree.Roots(active_collect_env_num, legal_actions)

    def _params(self):
        c = self._cfg
        return (c.pb_c_base, c.pb_c_init, c.discount_factor, c.value_delta_max)

    def search(self, roots: "mz_tree.Roots", model, latent_state_roots, to_play_batch: Union[int, List[Any]],
               task_id: Optional[int] = None) -> None:
        """mcts_ctree.py:267-368.  ``latent_state_roots``: np.ndarray or CUDA tensor [B,C,H,W]."""
        S = int(self._cfg.num_simulations)
        roots._materialize(S, self._params())     # reset + prepare on device, MinMax stats fresh (:291-292)
        t = roots._tree
        dev = roots.device
        if isinstance(latent_state_roots, torch.Tensor):
            lat = latent_state_roots.to(dev, torch.float32, non_blocking=True).contiguous()
        else:
            lat = torch.from_numpy(np.ascontiguousarray(latent_state_roots, dtype=np.float32)).to(dev, non_blocking=True)
        if isinstance(model, EfficientZeroModel):
            raise TypeError("MuZeroMCTSCtree.search: an EfficientZeroModel needs EfficientZeroMCTSCtree")
        if isinstance(model, (MuZeroModel, MuZeroModelMLP)):
            q = t.search_for(model, S)
            with torch.cuda.device(dev):
                cabi.check(t.lib.lz_search_run(q, lat.data_ptr(), int(self.deterministic), cabi.stream_ptr()),
                           "lz_search_run")
            self.last_num_kernels = t.lib.lz_search_num_kernels(q)
            return
        self._search_stepwise(roots, model, lat, S)

    def search_with_reuse(self, roots: "mz_tree.Roots", model, latent_state_roots, to_play_batch: Union[int, List[Any]],
                          true_action_list=None, reuse_value_list=None):
        """mcts_ctree.py:370-468 (ReZero): the root child of ``true_action`` is scored with the stored ``reuse_value`` and the
        descent stops there.  Returns ``(length, average_infer)`` like the reference: how many trees needed the network in
        the last simulation and on average.  One CUDA graph with a ``lightzero_b200`` model."""
        S = int(self._cfg.num_simulations)
        roots._materialize(S, self._params())
        t = roots._tree
        dev = roots.device
        if not isinstance(model, (MuZeroModel, MuZeroModelMLP)) or isinstance(model, EfficientZeroModel):
            raise NotImplementedError("search_with_reuse is fused only: pass a lightzero_b200 MuZeroModel / MuZeroModelMLP "
                                      "(or drive mz_tree.batch_traverse_with_reuse / batch_backpropagate_with_reuse yourself)")
        if isinstance(latent_state_roots, torch.Tensor):
            lat = latent_state_roots.to(dev, torch.float32, non_blocking=True).contiguous()
        else:
            lat = torch.from_numpy(np.ascontiguousarray(latent_state_roots, dtype=np.float32)).to(dev, non_blocking=True)
        B = roots.num
        ta = mz_tree._to_dev(true_action_list, torch.int32, dev, (B,))
        rv = mz_tree._to_dev(reuse_value_list, torch.float32, dev, (B,))
        counts = torch.empty(S, dtype=torch.int32, device=dev)
        cabi.check(t.lib.lz_tree_set_tiebreak(t.h, int(self.deterministic)), "lz_tree_set_tiebreak")   # the reference draws rand() % len(ties) (cnode.cpp:610-640)
        q = t.search_for(model, S)
        with torch.cuda.device(dev):
            cabi.check(t.lib.lz_search_run_with_reuse(q, lat.data_ptr(), ta.data_ptr(), rv.data_ptr(), counts.data_ptr(),
                                                      cabi.stream_ptr()), "lz_search_run_with_reuse")
        c = counts.cpu().numpy()
        return int(c[-1]), float(c.sum()) / S

    def _make_inverse_transforms(self, dev):
        """mcts_ctree.py:249-253: separate value and reward supports, both categorical (the only representation the CUDA
        transform implements)."""
        if self._inv is not None:
            return
        m = self._cfg.get("model", None)

        def rng(key):
            return tuple(m[key]) if m is not None and key in m else (-300., 301., 1.)
        if m is not None and not m.get("categorical_distribution", True):
            raise NotImplementedError("model.categorical_distribution=False: only the categorical (support) representation is implemented")
        self._inv = InverseScalarTransform(DiscreteSupport(*rng("value_support_range"), device=dev))
        vr, rr = rng("value_support_range"), rng("reward_support_range")
        self._inv_reward = self._inv if vr == rr else InverseScalarTransform(DiscreteSupport(*rr, device=dev))

    def _search_stepwise(self, roots, model, lat, S):
        t = roots._tree
        dev = roots.device
        self._make_inverse_transforms(dev)
        B = roots.num
        pool = torch.empty((S + 1,) + tuple(lat.shape), device=dev, dtype=torch.float32)
        pool[0] = lat
        rows = torch.arange(B, device=dev)
        with torch.no_grad(), torch.cuda.device(dev):
            if hasattr(model, "eval"):
                model.eval()
            for sim in range(S):
                self._traverse(t)
                latent_states = pool[t.ix.long(), rows]                       # mcts_ctree.py:323-324 on device
                out = model.recurrent_inference(latent_states, t.action.long())
                pool[sim + 1] = out.latent_state
                value = self._inv(out.value).reshape(-1).contiguous()        # :349 (value support)
                reward = self._inv_reward(out.reward).reshape(-1).contiguous()      # :350 (reward support)
                pol = out.policy_logits.to(torch.float32).contiguous()
                self._backpropagate(t, sim + 1, reward, value, pol)

    # the tree steps of _search_stepwise (GumbelMuZeroMCTSCtree swaps in the Gumbel descent and back-up)
    def _traverse(self, t):
        cabi.check(t.lib.lz_tree_traverse(t.h, int(self.deterministic), t.ix.data_ptr(), t.iy.data_ptr(),
                                          t.action.data_ptr(), t.search_len.data_ptr(), t.vtp.data_ptr(),
                                          cabi.stream_ptr()), "lz_tree_traverse")

    def _backpropagate(self, t, latent_index, reward, value, pol):
        cabi.check(t.lib.lz_tree_backpropagate(t.h, latent_index, reward.data_ptr(), value.data_ptr(),
                                               pol.data_ptr(), None, cabi.stream_ptr()), "lz_tree_backpropagate")


class EfficientZeroMCTSCtree(MuZeroMCTSCtree):
    """Mirror of ``lzero.mcts.tree_search.mcts_ctree.EfficientZeroMCTSCtree`` (mcts_ctree.py:671-876): same config keys
    (+ ``lstm_horizon_len``, read at :857), ``roots(n, legal_actions)`` and
    ``search(roots, model, latent_state_roots, reward_hidden_state_roots, to_play_batch)``.

    With a ``lightzero_b200.EfficientZeroModel`` the whole loop is one CUDA-graph launch (``lz_search_run_ez``): per
    simulation the descent (which also derives ``is_reset = search_len % lstm_horizon_len == 0``, :856-861), the conv
    trunk + prediction heads, the LSTM value-prefix head over all roots, and the back-up.  Any other model object is
    driven step-wise around the device trees.  Ties: first maximum (the reference's ``rand() % len(ties)`` with
    ``rand() == 0``; the EfficientZero tree has no deterministic switch, cnode.cpp:691)."""

    def __init__(self, cfg=None) -> None:
        super().__init__(cfg)
        self._cfg.setdefault("lstm_horizon_len", 5)
        # the reference tree has no deterministic switch (always rand() % len(ties)); here first maximum is the default (what the
        # parity tests pin) and ``deterministic=False`` in the config selects the uniform draw (lz_tree_set_tiebreak)
        self.deterministic = bool(self._cfg.get("deterministic", True))

    @classmethod
    def roots(cls, active_collect_env_num: int, legal_actions: List[Any]) -> "ez_tree.Roots":
        """mcts_ctree.py:715-727"""
        return ez_tree.Roots(active_collect_env_num, legal_actions)

    def search(self, roots: "ez_tree.Roots", model, latent_state_roots, reward_hidden_state_roots,
               to_play_batch: Union[int, List[Any]]) -> None:
        S, H = int(self._cfg.num_simulations), int(self._cfg.lstm_horizon_len)
        assert H > 0                                   # mcts_ctree.py:857
        roots._ez, roots._lstm_horizon = True, H
        roots._materialize(S, self._params())
        t = roots._tree
        dev = roots.device
        cabi.check(t.lib.lz_tree_set_tiebreak(t.h, int(self.deterministic)), "lz_tree_set_tiebreak")

        def dev_f32(x):
            if isinstance(x, torch.Tensor):
                return x.to(dev, torch.float32, non_blocking=True).contiguous()
            return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev, non_blocking=True)
        lat = dev_f32(latent_state_roots)
        B = roots.num
        h0 = dev_f32(reward_hidden_state_roots[0]).reshape(B, -1)
        h1 = dev_f32(reward_hidden_state_roots[1]).reshape(B, -1)
        if isinstance(model, EfficientZeroModel):
            q = t.search_for(model, S, (1, H))
            with torch.cuda.device(dev):
                cabi.check(t.lib.lz_search_run_ez(q, lat.data_ptr(), h0.data_ptr(), h1.data_ptr(), cabi.stream_ptr()),
                           "lz_search_run_ez")
            self.last_num_kernels = t.lib.lz_search_num_kernels(q)
            return
        self._search_stepwise_ez(roots, model, lat, h0, h1, S, H)

    def search_with_reuse(self, roots: "ez_tree.Roots", model, latent_state_roots, reward_hidden_state_roots,
                          to_play_batch: Union[int, List[Any]], true_action_list=None, reuse_value_list=None):
        """mcts_ctree.py:878-1003 (ReZero on the EfficientZero trees) as one CUDA graph (``lz_search_run_ez_with_reuse``); returns
        ``(length, average_infer)`` like the reference.  Fused only: other model objects drive
        ``ez_tree.batch_traverse_with_reuse`` / ``batch_backpropagate_with_reuse`` themselves."""
        S, H = int(self._cfg.num_simulations), int(self._cfg.lstm_horizon_len)
        assert H > 0
        if not isinstance(model, EfficientZeroModel):
            raise NotImplementedError("EfficientZeroMCTSCtree.search_with_reuse is fused only: pass a lightzero_b200 EfficientZeroModel")
        roots._ez, roots._lstm_horizon = True, H
        roots._materialize(S, self._params())
        t = roots._tree
        dev = roots.device
        cabi.check(t.lib.lz_tree_set_tiebreak(t.h, int(self.deterministic)), "lz_tree_set_tiebreak")

        def dev_f32(x):
            if isinstance(x, torch.Tensor):
                return x.to(dev, torch.float32, non_blocking=True).contiguous()
            return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev, non_blocking=True)
        lat = dev_f32(latent_state_roots)
        B = roots.num
        h0 = dev_f32(reward_hidden_state_roots[0]).reshape(B, -1)
        h1 = dev_f32(reward_hidden_state_roots[1]).reshape(B, -1)
        ta = mz_tree._to_dev(true_action_list, torch.int32, dev, (B,))
        rv = mz_tree._to_dev(reuse_value_list, torch.float32, dev, (B,))
        counts = torch.empty(S, dtype=torch.int32, device=dev)
        q = t.search_for(model, S, (1, H))
        with torch.cuda.device(dev):
            cabi.check(t.lib.lz_search_run_ez_with_reuse(q, lat.data_ptr(), h0.data_ptr(), h1.data_ptr(), ta.data_ptr(), rv.data_ptr(),
                                                         counts.data_ptr(), cabi.stream_ptr()), "lz_search_run_ez_with_reuse")
        c = counts.cpu().numpy()
        return int(c[-1]), float(c.sum()) / S

    def _search_stepwise_ez(self, roots, model, lat, h0, h1, S, H):
        t = roots._tree
        dev = roots.device
        self._make_inverse_transforms(dev)
        B = roots.num
        pool = torch.empty((S + 1,) + tuple(lat.shape), device=dev, dtype=torch.float32)
        hp0 = torch.zeros((S + 1, B, h0.shape[1]), device=dev)
        hp1 = torch.zeros((S + 1, B, h1.shape[1]), device=dev)
        pool[0], hp0[0], hp1[0] = lat, h0, h1
        rows = torch.arange(B, device=dev)
        reset = torch.empty(B, dtype=torch.int32, device=dev)
        with torch.no_grad(), torch.cuda.device(dev):
            if hasattr(model, "eval"):
                model.eval()
            for sim in range(S):
                cabi.check(t.lib.lz_tree_traverse_ez(t.h, t.ix.data_ptr(), t.iy.data_ptr(), t.action.data_ptr(),
                                                     t.search_len.data_ptr(), t.vtp.data_ptr(), reset.data_ptr(),
                                                     cabi.stream_ptr()), "lz_tree_traverse_ez")
                ix = t.ix.long()
                hidden = (hp0[ix, rows].unsqueeze(0), hp1[ix, rows].unsqueeze(0))          # mcts_ctree.py:819-831
                out = model.recurrent_inference(pool[ix, rows], hidden, t.action.long())
                pool[sim + 1] = out.latent_state
                keep = (reset == 0).to(torch.float32).unsqueeze(1)                          # :856-863
                hp0[sim + 1] = out.reward_hidden_state[0].reshape(B, -1) * keep
                hp1[sim + 1] = out.reward_hidden_state[1].reshape(B, -1) * keep
                value = self._inv(out.value).reshape(-1).contiguous()
                vprefix = self._inv_reward(out.value_prefix).reshape(-1).contiguous()
                pol = out.policy_logits.to(torch.float32).contiguous()
                cabi.check(t.lib.lz_tree_backpropagate_ez(t.h, sim + 1, vprefix.data_ptr(), value.data_ptr(), pol.data_ptr(),
                                                          reset.data_ptr(), None, cabi.stream_ptr()),
                           "lz_tree_backpropagate_ez")


class UniZeroMCTSCtree(MuZeroMCTSCtree):
    """Mirror of ``lzero.mcts.tree_search.mcts_ctree.UniZeroMCTSCtree`` (mcts_ctree.py:19-208): the MuZero tree unchanged
    (``mz_tree.Roots``, :64-75), ``deterministic`` taken from the config (default False, :41-42, passed to ``batch_traverse``
    at :128-137), and a world model that is called with the whole search history:
    ``model.recurrent_inference(state_action_history, simulation_index, search_depth[, timestep | task_id=...])`` (:160-176),
    where ``state_action_history`` is the list of ``(latent_states ndarray, last_actions LongTensor)`` of every simulation so far
    (:147) -- the UniZero transformer re-derives its KV cache from it.  ``search`` returns ``first_action_latent_map`` (:90, :183-189).

    The DRIVER is what this class provides: the trees stay on the GPU (device ``batch_traverse`` / ``batch_backpropagate``), the
    history hand-off follows the reference's host-array contract (one D2H of the gathered latents / actions / search depths per
    simulation, exactly what the reference's own loop does at :144-147).  The transformer world model itself (``WorldModel`` with
    its KV cache, lzero/model/unizero_world_models/) is NOT part of this library: pass the reference's model object, or any
    object with that ``recurrent_inference`` signature."""

    config = dict(MuZeroMCTSCtree.config, deterministic=False)     # mcts_ctree.py:28-43

    def search(self, roots: "mz_tree.Roots", model, latent_state_roots, to_play_batch: Union[int, List[Any]],
               timestep: Union[int, List[Any]] = None, task_id: Optional[int] = None) -> dict:
        S = int(self._cfg.num_simulations)
        roots._materialize(S, self._params())
        t = roots._tree
        dev = roots.device
        self._make_inverse_transforms(dev)
        B = roots.num
        lat0 = latent_state_roots.detach().cpu().numpy() if isinstance(latent_state_roots, torch.Tensor) else np.asarray(latent_state_roots)
        latent_pool = [np.ascontiguousarray(lat0, dtype=np.float32)]
        first_action_latent_map = {env_id: {} for env_id in range(B)}
        state_action_history = []
        with torch.no_grad(), torch.cuda.device(dev):
            if hasattr(model, "eval"):
                model.eval()
            for simulation_index in range(S):
                cabi.check(t.lib.lz_tree_traverse(t.h, int(self.deterministic), t.ix.data_ptr(), t.iy.data_ptr(),
                                                  t.action.data_ptr(), t.search_len.data_ptr(), t.vtp.data_ptr(),
                                                  cabi.stream_ptr()), "lz_tree_traverse")
                ix, iy = t.ix.cpu().numpy(), t.iy.cpu().numpy()
                last_actions = t.action.cpu().long()
                search_depth = t.search_len.cpu().numpy().tolist()
                latent_states = np.stack([latent_pool[x][y] for x, y in zip(ix, iy)])          # :141-144
                state_action_history.append((latent_states, last_actions.to(self._cfg.device)))  # :147
                if timestep is None:                                                            # :160-176
                    if task_id is not None:
                        out = model.recurrent_inference(state_action_history, simulation_index, search_depth, task_id=task_id)
                    else:
                        out = model.recurrent_inference(state_action_history, simulation_index, search_depth)
                else:
                    if task_id is not None:
                        out = model.recurrent_inference(state_action_history, simulation_index, search_depth, task_id=task_id)
                    else:
                        out = model.recurrent_inference(state_action_history, simulation_index, search_depth, timestep)
                latent = out.latent_state.detach().cpu().numpy() if isinstance(out.latent_state, torch.Tensor) else np.asarray(out.latent_state)
                value = self._inv(out.value.to(dev)).reshape(-1).contiguous()                   # :180
                reward = self._inv_reward(out.reward.to(dev)).reshape(-1).contiguous()          # :181
                pol = out.policy_logits.to(dev, torch.float32).contiguous()
                for env_id in range(B):                                                         # :183-189
                    a = int(last_actions[env_id].item())
                    if search_depth[env_id] == 1 and a not in first_action_latent_map[env_id]:
                        first_action_latent_map[env_id][a] = latent[env_id]
                latent_pool.append(latent)
                cabi.check(t.lib.lz_tree_backpropagate(t.h, simulation_index + 1, reward.data_ptr(), value.data_ptr(),
                                                       pol.data_ptr(), None, cabi.stream_ptr()), "lz_tree_backpropagate")
        return first_action_latent_map


class GumbelMuZeroMCTSCtree(MuZeroMCTSCtree):
    """Mirror of ``lzero.mcts.tree_search.mcts_ctree.GumbelMuZeroMCTSCtree`` (mcts_ctree.py:1005-1174): same class-level
    ``config``, ``default_config()``, ``roots(n, legal_actions)`` (``gmz_tree.Roots``) and
    ``search(roots, model, latent_state_roots, to_play_batch)``; ``num_simulations``, ``max_num_considered_actions`` and
    ``discount_factor`` come from the policy config as in the reference (defaults of gumbel_muzero.py: 4 and 0.997).

    With a ``lightzero_b200`` MuZeroModel / MuZeroModelMLP the whole search is one CUDA-graph launch (``lz_search_run_gumbel``);
    any other model object is driven step-wise around the device trees.  Root choice is sequential halving over the fixed
    Gumbel draw and interior choice the completed-Q improved policy: no random numbers, so both modes reproduce the reference
    tree bit for bit on the same network outputs."""

    # mcts_ctree.py:1018-1027
    config = dict(
        num_simulations=50,
        root_dirichlet_alpha=0.3,
        root_noise_weight=0.25,
        value_delta_max=0.01,
    )

    def __init__(self, cfg=None) -> None:
        super().__init__(cfg)
        self._cfg.setdefault("max_num_considered_actions", 4)
        self._cfg.setdefault("env_type", "not_board_games")

    @classmethod
    def roots(cls, active_collect_env_num: int, legal_actions: List[Any]) -> "gmz_tree.Roots":
        """mcts_ctree.py:1062-1074"""
        return gmz_tree.Roots(active_collect_env_num, legal_actions)

    def _gumbel_params(self):
        return int(self._cfg.num_simulations), int(self._cfg.max_num_considered_actions)

    def search(self, roots: "gmz_tree.Roots", model, latent_state_roots, to_play_batch: Union[int, List[Any]]) -> None:
        """mcts_ctree.py:1076-1174.  ``latent_state_roots``: np.ndarray or CUDA tensor [B, ...]."""
        S, m = self._gumbel_params()
        roots._materialize(S, (S, m))        # reset + Gumbel tables + prepare on the device
        t = roots._tree
        dev = roots.device
        if isinstance(latent_state_roots, torch.Tensor):
            lat = latent_state_roots.to(dev, torch.float32, non_blocking=True).contiguous()
        else:
            lat = torch.from_numpy(np.ascontiguousarray(latent_state_roots, dtype=np.float32)).to(dev, non_blocking=True)
        if isinstance(model, EfficientZeroModel):
            raise TypeError("GumbelMuZeroMCTSCtree.search: Gumbel MuZero runs on MuZero models, not an EfficientZeroModel")
        if isinstance(model, (MuZeroModel, MuZeroModelMLP)):
            q = t.search_for(model, S)
            with torch.cuda.device(dev):
                cabi.check(t.lib.lz_search_run_gumbel(q, lat.data_ptr(), float(self._cfg.discount_factor), cabi.stream_ptr()),
                           "lz_search_run_gumbel")
            self.last_num_kernels = t.lib.lz_search_num_kernels(q)
            return
        self._search_stepwise(roots, model, lat, S)

    def _traverse(self, t):
        cabi.check(t.lib.lz_tree_traverse_gumbel(t.h, float(self._cfg.discount_factor), t.ix.data_ptr(), t.iy.data_ptr(),
                                                 t.action.data_ptr(), t.search_len.data_ptr(), t.vtp.data_ptr(),
                                                 cabi.stream_ptr()), "lz_tree_traverse_gumbel")

    def _backpropagate(self, t, latent_index, reward, value, pol):
        cabi.check(t.lib.lz_tree_backpropagate_gumbel(t.h, latent_index, float(self._cfg.discount_factor), reward.data_ptr(),
                                                      value.data_ptr(), pol.data_ptr(), cabi.stream_ptr()),
                   "lz_tree_backpropagate_gumbel")
