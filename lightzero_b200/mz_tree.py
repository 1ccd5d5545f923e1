"""Device-resident mirror of the reference's Cython module ``lzero.mcts.ctree.ctree_muzero.mz_tree``
(mz_tree.pyx:5-107): ``Roots``, ``MinMaxStatsList``, ``ResultsWrapper``, ``batch_traverse``,
``batch_backpropagate`` with the same names, argument order and meaning.  Every list argument may
also be a numpy array or a CUDA tensor (which avoids the host round trip).  State lives in the CUDA
trees behind ``lz_tree_*`` (include/lzb200.h); nothing here computes on the CPU.

Differences a caller can observe:
  * list outputs are materialised with ONE device->host copy when asked for (``get_distributions``,
    ``get_values``, the tuple returned by ``batch_traverse``); ``*_tensor`` variants stay on device;
  * ``MinMaxStatsList`` is bookkeeping only -- min/max live inside the tree and are reset when the
    Roots are (re)prepared, i.e. once per search like mcts_ctree.py:291-292.
"""
import threading
from typing import List, Optional

import numpy as np
import torch

from . import cabi

DEFAULT_MAX_SIMS = 64     # node-pool capacity when a Roots is driven step-wise without a known budget
_tree_pool = {}           # (device index, B, A, max_sims) -> [TreeHandle]
_pool_lock = threading.Lock()


class TreeHandle:
    """Owns one lz_tree (+ lazily one lz_search per model) and its scratch tensors."""

    def __init__(self, device, B, A, max_sims):
        self.device, self.B, self.A, self.max_sims = device, B, A, max_sims
        self.lib = cabi.load()
        h = cabi.c_void_p()
        with torch.cuda.device(device):
            cabi.check(self.lib.lz_tree_create(B, A, max_sims, h), "lz_tree_create")
        self.h = h
        self.busy = False
        self.params = None
        i32 = dict(dtype=torch.int32, device=device)
        self.ix, self.iy, self.action = (torch.empty(B, **i32) for _ in range(3))
        self.search_len, self.vtp = torch.empty(B, **i32), torch.empty(B, **i32)
        self.visits = torch.empty(B, A, **i32)
        self.nlegal = torch.empty(B, **i32)
        self.values = torch.empty(B, dtype=torch.float32, device=device)
        self.traj = torch.empty(B, max_sims + 1, **i32)
        self.searches = {}    # (model serial, num_simulations, mode...) -> lz_search handle; dropped when the model dies

    def set_params(self, pb_c_base, pb_c_init, discount, delta):
        p = (int(pb_c_base), float(pb_c_init), float(discount), float(delta))
        if p != self.params:
            with torch.cuda.device(self.device):
                cabi.check(self.lib.lz_tree_set_params(self.h, *p), "lz_tree_set_params")
            self.params = p

    def search_for(self, model, num_simulations, mode=()):
        # keyed by the model's serial (unique for the life of the process; id() is recycled after garbage collection).  The
        # captured graph is re-captured inside the library when the model's weights / math mode or this tree's parameters
        # change (generation counters, csrc/search.cu), so one lz_search per (model, num_simulations, mode) is enough
        key = (model._serial, num_simulations) + tuple(mode)     # mode: (ez, lstm_horizon_len)
        if key not in self.searches:
            q = cabi.c_void_p()
            with torch.cuda.device(self.device):
                cabi.check(self.lib.lz_search_create(self.h, model._h, num_simulations, q), "lz_search_create")
            self.searches[key] = q
        return self.searches[key]

    def __del__(self):
        try:
            for q in self.searches.values():
                self.lib.lz_search_destroy(q)
            self.lib.lz_tree_destroy(self.h)
        except Exception:
            pass


def acquire_tree(device, B, A, max_sims) -> TreeHandle:
    key = (device.index, B, A, max_sims)
    with _pool_lock:
        for h in _tree_pool.setdefault(key, []):
            if not h.busy:
                h.busy = True
                return h
        h = TreeHandle(device, B, A, max_sims)
        h.busy = True
        _tree_pool[key].append(h)
        return h


def drop_model_searches(serial: int):
    """Called when a model wrapper is destroyed: destroys every lz_search bound to that lz_model (they hold its pointer and
    graphs captured against its device tables)."""
    with _pool_lock:
        handles = [h for hs in _tree_pool.values() for h in hs]
    for h in handles:
        for key in [k for k in h.searches if k[0] == serial]:
            q = h.searches.pop(key)
            try:
                h.lib.lz_search_destroy(q)
            except Exception:
                pass


def _to_dev(x, dtype, device, shape=None):
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        t = x.to(device=device, dtype=dtype, non_blocking=True)
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype={torch.float32: np.float32, torch.int32: np.int32,
                                                                       torch.uint8: np.uint8}[dtype]))).to(device, non_blocking=True)
    if shape is not None:
        t = t.reshape(shape)
    return t.contiguous()


class MinMaxStatsList:
    """mz_tree.pyx:5-15"""

    def __init__(self, num: int):
        self.num = num
        self.value_delta_max = 0.0

    def set_delta(self, value_delta_max: float):
        self.value_delta_max = float(value_delta_max)


class ResultsWrapper:
    """mz_tree.pyx:17-24"""

    def __init__(self, num: int):
        self.num = num
        self._roots = None

    def get_search_len(self) -> List[int]:
        return self._roots._tree.search_len.cpu().tolist()


class Roots:
    """mz_tree.pyx:26-59.  ``legal_actions_list``: list of lists (any order), or a uint8/bool mask
    tensor/array [root_num, A]."""

    def __init__(self, root_num: int, legal_actions_list, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("lightzero_b200.mz_tree.Roots needs a CUDA device; there is no CPU fallback")
        self.root_num = root_num
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._legal_lists = None
        self._mask = None
        self._mask_dev = None
        if isinstance(legal_actions_list, (torch.Tensor, np.ndarray)) and np.ndim(legal_actions_list) == 2 and \
                str(legal_actions_list.dtype).split(".")[-1] in ("uint8", "bool"):
            self._mask = legal_actions_list
        else:
            self._legal_lists = [list(l) for l in legal_actions_list]
            assert len(self._legal_lists) == root_num
        self._pending = None      # prepare() arguments until the tree is materialised
        self._ez, self._lstm_horizon = False, 5     # EfficientZero value-prefix semantics (set by ez_tree.Roots)
        self._tree: Optional[TreeHandle] = None
        self._delta_reset = None

    # ---- reference API ---------------------------------------------------------------------------
    def prepare(self, root_noise_weight: float, noises, value_prefix_pool, policy_logits_pool, to_play_batch):
        self._stage(float(root_noise_weight), noises, value_prefix_pool, policy_logits_pool, to_play_batch)

    def prepare_no_noise(self, value_prefix_pool, policy_logits_pool, to_play_batch):
        self._stage(0.0, None, value_prefix_pool, policy_logits_pool, to_play_batch)

    def get_distributions(self) -> List[List[int]]:
        v, n = self.get_distributions_tensor()
        v, n = v.cpu().numpy(), n.cpu().numpy()
        return [v[i, :n[i]].tolist() for i in range(self.root_num)]

    def get_values(self) -> List[float]:
        return self.get_values_tensor().cpu().tolist()

    def get_trajectories(self) -> List[List[int]]:
        t = self._need_tree()
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_results(t.h, None, None, None, t.traj.data_ptr(), cabi.stream_ptr()), "lz_tree_results")
        tr = t.traj.cpu().numpy()
        return [row[row >= 0].tolist() for row in tr]

    def clear(self):
        if self._tree is not None:
            self._tree.busy = False
            self._tree = None

    @property
    def num(self) -> int:
        return self.root_num

    def __del__(self):
        try:
            self.clear()
        except Exception:
            pass

    # ---- device-side extras ----------------------------------------------------------------------
    def get_distributions_tensor(self):
        """(visits int32 [B,A] in legal order, -1 padded; nlegal int32 [B]) on device."""
        t = self._need_tree()
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_results(t.h, t.visits.data_ptr(), t.values.data_ptr(), t.nlegal.data_ptr(), None,
                                             cabi.stream_ptr()), "lz_tree_results")
        return t.visits, t.nlegal

    def select_action_tensor(self, temperature: float = 1.0, deterministic: bool = False, seed: int = 0):
        """lzero/policy/utils.py:637-661 for every root on the device -> (action id, position in the legal list, entropy)."""
        t = self._need_tree()
        act = torch.empty(self.root_num, dtype=torch.int32, device=self.device)
        pos = torch.empty(self.root_num, dtype=torch.int32, device=self.device)
        ent = torch.empty(self.root_num, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_select_action(t.h, float(temperature), int(bool(deterministic)), int(seed) & (2 ** 64 - 1),
                                                   act.data_ptr(), pos.data_ptr(), ent.data_ptr(), cabi.stream_ptr()),
                       "lz_tree_select_action")
        return act, pos, ent

    def get_values_tensor(self):
        t = self._need_tree()
        with torch.cuda.device(self.device):
            cabi.check(t.lib.lz_tree_results(t.h, None, t.values.data_ptr(), None, None, cabi.stream_ptr()), "lz_tree_results")
        return t.values

    # ---- internals -------------------------------------------------------------------------------
    def _stage(self, w, noises, rewards, policies, to_play):
        B = self.root_num
        pol = _to_dev(policies, torch.float32, self.device)
        pol = pol.reshape(B, -1).contiguous()
        A = pol.shape[1]
        nz = None
        if noises is not None:
            if isinstance(noises, (torch.Tensor, np.ndarray)):
                nz = _to_dev(noises, torch.float32, self.device, (B, A))
            else:   # list of per-root lists in legal order (policy/muzero.py:763-766)
                arr = np.zeros((B, A), np.float32)
                for i, n in enumerate(noises):
                    arr[i, :len(n)] = n
                nz = torch.from_numpy(arr).to(self.device, non_blocking=True)
        rew = None
        if rewards is not None and not (isinstance(rewards, list) and all(r == 0 for r in rewards)):
            rew = _to_dev(rewards, torch.float32, self.device, (B,))
        tp = _to_dev(to_play, torch.int32, self.device, (B,)) if to_play is not None else None
        self._pending = dict(w=w, noise=nz, rewards=rew, logits=pol, to_play=tp, A=A)
        if self._tree is not None:      # re-prepare of an already materialised tree
            self._materialize(self._tree.max_sims)

    def _need_tree(self) -> TreeHandle:
        if self._tree is None:
            self._materialize(DEFAULT_MAX_SIMS)
        return self._tree

    def _materialize(self, max_sims: int, params=None):
        if self._pending is None:
            raise RuntimeError("Roots: prepare()/prepare_no_noise() has not been called")
        p = self._pending
        A = p["A"]
        if self._tree is not None and (self._tree.max_sims < max_sims or self._tree.A != A):
            self.clear()
        if self._tree is None:
            self._tree = acquire_tree(self.device, self.root_num, A, max_sims)
        t = self._tree
        if params is not None:
            t.set_params(*params)
        s = None
        with torch.cuda.device(self.device):
            s = cabi.stream_ptr()
            cabi.check(t.lib.lz_tree_set_ez(t.h, int(self._ez), int(self._lstm_horizon)), "lz_tree_set_ez")
            if self._mask is not None:
                if self._mask_dev is None:      # uploaded once per Roots, not once per search
                    self._mask_dev = _to_dev(self._mask, torch.uint8, self.device, (self.root_num, A))
                cabi.check(t.lib.lz_tree_reset_mask(t.h, self._mask_dev.data_ptr(), s), "lz_tree_reset_mask")
            else:
                identity = list(range(A))
                if all(l == identity for l in self._legal_lists):
                    cabi.check(t.lib.lz_tree_reset(t.h, None, None, s), "lz_tree_reset")
                else:
                    legal = np.full((self.root_num, A), -1, np.int32)
                    nl = np.zeros(self.root_num, np.int32)
                    for i, l in enumerate(self._legal_lists):
                        nl[i] = len(l)
                        legal[i, :len(l)] = l
                    dl = torch.from_numpy(legal).to(self.device)
                    dn = torch.from_numpy(nl).to(self.device)
                    cabi.check(t.lib.lz_tree_reset(t.h, dl.data_ptr(), dn.data_ptr(), s), "lz_tree_reset")
                    self._keep = (dl, dn)
            self._prepare_tree(t, p, s)

    def _prepare_tree(self, t: TreeHandle, p: dict, s):
        """Expands the roots of the freshly reset tree from the staged prepare() arguments."""
        cabi.check(t.lib.lz_tree_prepare(t.h, p["logits"].data_ptr(), cabi.ptr(p["noise"]), p["w"],
                                         cabi.ptr(p["rewards"]), cabi.ptr(p["to_play"]), s), "lz_tree_prepare")


def batch_traverse(roots: Roots, pb_c_base: int, pb_c_init: float, discount_factor: float,
                   min_max_stats_lst: MinMaxStatsList, results: ResultsWrapper, virtual_to_play_batch,
                   deterministic: bool = False, return_tensors: bool = False):
    """mz_tree.pyx:94-99 -> (latent_state_index_in_search_path, latent_state_index_in_batch, last_actions,
    virtual_to_play_batch)."""
    if roots._tree is None:
        roots._materialize(DEFAULT_MAX_SIMS)
    t = roots._tree
    t.set_params(pb_c_base, pb_c_init, discount_factor, min_max_stats_lst.value_delta_max)
    with torch.cuda.device(roots.device):
        cabi.check(t.lib.lz_tree_traverse(t.h, int(bool(deterministic)), t.ix.data_ptr(), t.iy.data_ptr(),
                                          t.action.data_ptr(), t.search_len.data_ptr(), t.vtp.data_ptr(),
                                          cabi.stream_ptr()), "lz_tree_traverse")
    results._roots = roots
    if return_tensors:
        return t.ix, t.iy, t.action, t.vtp
    packed = torch.stack((t.ix, t.iy, t.action, t.vtp)).cpu().numpy()
    return packed[0].tolist(), packed[1].tolist(), packed[2].tolist(), packed[3].tolist()


def batch_backpropagate(current_latent_state_index: int, discount_factor: float, value_prefixs, values, policies,
                        min_max_stats_lst: MinMaxStatsList, results: ResultsWrapper, to_play_batch):
    """mz_tree.pyx:73-82"""
    roots = results._roots
    t = roots._tree
    B, A = roots.root_num, t.A
    dev = roots.device
    rew = _to_dev(value_prefixs, torch.float32, dev, (B,))
    val = _to_dev(values, torch.float32, dev, (B,))
    pol = _to_dev(policies, torch.float32, dev, (B, A))
    tp = _to_dev(to_play_batch, torch.int32, dev, (B,)) if to_play_batch is not None else None
    with torch.cuda.device(dev):
        cabi.check(t.lib.lz_tree_backpropagate(t.h, int(current_latent_state_index), rew.data_ptr(), val.data_ptr(),
                                               pol.data_ptr(), cabi.ptr(tp), cabi.stream_ptr()),
                   "lz_tree_backpropagate")
    t._keep = (rew, val, pol, tp)


def batch_traverse_with_reuse(roots: Roots, pb_c_base: int, pb_c_init: float, discount_factor: float,
                              min_max_stats_lst: MinMaxStatsList, results: ResultsWrapper, virtual_to_play_batch,
                              true_action, reuse_value, return_tensors: bool = False):
    """mz_tree.pyx batch_traverse_with_reuse (cnode.cpp:828-932): ``latent_state_index_in_search_path`` is -1 for trees
    that stopped on an already expanded child of the root (no inference needed)."""
    if roots._tree is None:
        roots._materialize(DEFAULT_MAX_SIMS)
    t = roots._tree
    t.set_params(pb_c_base, pb_c_init, discount_factor, min_max_stats_lst.value_delta_max)
    dev = roots.device
    ta = _to_dev(true_action, torch.int32, dev, (roots.root_num,))
    rv = _to_dev(reuse_value, torch.float32, dev, (roots.root_num,))
    with torch.cuda.device(dev):
        cabi.check(t.lib.lz_tree_traverse_with_reuse(t.h, ta.data_ptr(), rv.data_ptr(), t.ix.data_ptr(), t.iy.data_ptr(),
                                                     t.action.data_ptr(), t.search_len.data_ptr(), t.vtp.data_ptr(),
                                                     cabi.stream_ptr()), "lz_tree_traverse_with_reuse")
    results._roots = roots
    t._keep = (ta, rv)
    if return_tensors:
        return t.ix, t.iy, t.action, t.vtp
    packed = torch.stack((t.ix, t.iy, t.action, t.vtp)).cpu().numpy()
    return packed[0].tolist(), packed[1].tolist(), packed[2].tolist(), packed[3].tolist()


def batch_backpropagate_with_reuse(current_latent_state_index: int, discount_factor: float, value_prefixs, values, policies,
                                   min_max_stats_lst: MinMaxStatsList, results: ResultsWrapper, to_play_batch,
                                   no_inference_lst, reuse_lst, reuse_value_lst, _is_reset_list=None):
    """mz_tree.pyx batch_backpropagate_with_reuse (cnode.cpp:502-549).  ``value_prefixs`` / ``values`` / ``policies`` are the
    COMPACTED network outputs of the trees that were inferred (the driver skips the others, mcts_ctree.py:424-432);
    they are scattered back to per-tree rows here, using ``no_inference_lst`` exactly as the C++ loop consumes it."""
    roots = results._roots
    t = roots._tree
    B, A = roots.root_num, t.A
    dev = roots.device
    skip = np.zeros(B, bool)
    skip[[i for i in no_inference_lst if i >= 0]] = True
    rank = np.cumsum(~skip) - 1                     # compact row of every inferred tree
    rank[skip] = -1
    n = int((~skip).sum())
    idx = torch.from_numpy(np.nonzero(~skip)[0]).to(dev)

    def scatter(x, shape):
        full = torch.zeros((B,) + shape, device=dev, dtype=torch.float32)
        if n:
            full[idx] = _to_dev(x, torch.float32, dev, (n,) + shape)
        return full
    rew, val, pol = scatter(value_prefixs, ()), scatter(values, ()), scatter(policies, (A,))
    rv = _to_dev(reuse_value_lst, torch.float32, dev, (B,))
    rk = torch.from_numpy(rank.astype(np.int32)).to(dev)
    tp = _to_dev(to_play_batch, torch.int32, dev, (B,)) if to_play_batch is not None else None
    rs = _to_dev(_is_reset_list, torch.int32, dev, (B,)) if _is_reset_list is not None else None
    with torch.cuda.device(dev):
        cabi.check(t.lib.lz_tree_backpropagate_with_reuse(t.h, int(current_latent_state_index), rew.data_ptr(), val.data_ptr(),
                                                          pol.data_ptr(), rv.data_ptr(), rk.data_ptr(), cabi.ptr(rs), cabi.ptr(tp),
                                                          cabi.stream_ptr()), "lz_tree_backpropagate_with_reuse")
    t._keep = (rew, val, pol, rv, rk, rs, tp)
