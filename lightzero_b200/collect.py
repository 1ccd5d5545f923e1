"""Mirror of the search-driving part of ``MuZeroPolicy._forward_collect`` / ``_forward_eval``
(lzero/policy/muzero.py:705-829, 872-956) and of ``select_action`` (lzero/policy/utils.py:637-661).

``MuZeroCollectPolicy.forward_collect(obs, action_mask, temperature, to_play)`` takes what the
reference's collector passes (a stacked observation batch, a 0/1 action mask, to_play) and returns
the same per-environment output dict.  Observations may live in (pinned) HOST memory: the copy to the
device, the representation+prediction networks, root preparation with Dirichlet noise, the whole
num_simulations search (one CUDA graph) and the result read-back are issued back to back on one
stream; the only host synchronisation is the final read of the results.
"""
from typing import Dict, List, Optional

import numpy as np
import torch

from . import cabi, mz_tree
from .efficientzero_model import EfficientZeroModel
from .mcts_ctree import EfficientZeroMCTSCtree, MuZeroMCTSCtree
from .muzero_model import MuZeroModel


def select_action(visit_counts: np.ndarray, temperature: float = 1, deterministic: bool = True):
    """lzero/policy/utils.py:637-661 (same arithmetic, fp64 numpy)."""
    action_probs = [visit_count_i ** (1 / temperature) for visit_count_i in visit_counts]
    action_probs = [x / sum(action_probs) for x in action_probs]
    if deterministic:
        action_pos = int(np.argmax([v for v in visit_counts]))
    else:
        action_pos = int(np.random.choice(len(visit_counts), p=action_probs))
    p = np.asarray(action_probs, np.float64)
    nz = p[p > 0]
    entropy = float(-(nz * np.log(nz)).sum() / np.log(2.0))   # scipy.stats.entropy(action_probs, base=2): natural-log entropy / ln 2
    return action_pos, entropy


class MuZeroCollectPolicy:
    def __init__(self, model: MuZeroModel, cfg: Optional[dict] = None):
        self.model = model
        self.mcts = MuZeroMCTSCtree(cfg or {})
        self.cfg = self.mcts._cfg
        self.device = model.device
        self._buf = {}
        self.h2d_chunks = 2      # host observation batches are copied in this many overlapped pieces
        self._tree_mode = (0, 5)   # (EfficientZero value-prefix trees?, lstm_horizon_len)

    # ---- device-resident fast path ---------------------------------------------------------------
    def _bufs(self, B, A):
        key = (B, A)
        if key not in self._buf:
            d = self.device
            self._buf[key] = dict(
                pred_value=torch.empty(B, device=d), logits=torch.empty(B, A, device=d),
                obs=None, mask=torch.empty(B, A, dtype=torch.uint8, device=d), noise=torch.empty(B, A, device=d),
                to_play=torch.empty(B, dtype=torch.int32, device=d),
                h_visits=torch.empty(B, A, dtype=torch.int32).pin_memory(),
                h_values=torch.empty(B).pin_memory(), h_pred=torch.empty(B).pin_memory(),
                h_logits=torch.empty(B, A).pin_memory(), h_nlegal=torch.empty(B, dtype=torch.int32).pin_memory(),
                action=torch.empty(B, dtype=torch.int32, device=d), action_pos=torch.empty(B, dtype=torch.int32, device=d),
                entropy=torch.empty(B, device=d), h_action=torch.empty(B, dtype=torch.int32).pin_memory(),
                h_entropy=torch.empty(B).pin_memory())
        return self._buf[key]

    def search_batch(self, obs: torch.Tensor, action_mask, noises, to_play=None, deterministic=None,
                     read_back: bool = True, select=None):
        """obs [B,C,H,W] (host or device), action_mask [B,A] 0/1, noises [B,A] rows in legal order or None
        (eval).  Returns dict of tensors; with read_back=True they are pinned host tensors and the call
        ends with the single stream synchronisation of the step.  select=(temperature, deterministic_action, seed) also
        runs select_action (policy/utils.py:637-661) on the device and returns 'action' / 'entropy'."""
        B = obs.shape[0]
        A = self.model.action_space_size
        S = int(self.cfg.num_simulations)
        bufs = self._bufs(B, A)
        dev = self.device
        det = self.mcts.deterministic if deterministic is None else bool(deterministic)
        with torch.cuda.device(dev):
            host_path = not obs.is_cuda
            # uint8 frames (what the Atari emulator delivers) stay uint8 on the wire: a quarter of the bytes; the [0, 1] scaling
            # of the reference's ScaledFloatFrameWrapper happens inside the first conv kernel (lz_search_collect*_u8)
            u8 = obs.dtype == torch.uint8
            if host_path:
                h_obs = obs.contiguous() if u8 else obs.to(torch.float32).contiguous()
                h_mask = (action_mask if isinstance(action_mask, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(action_mask))).to(torch.uint8).contiguous()
                h_noise = None
                if noises is not None:
                    h_noise = (noises if isinstance(noises, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(noises, dtype=np.float32))).to(torch.float32).contiguous()
                h_tp = None
                if to_play is not None:
                    h_tp = (to_play if isinstance(to_play, torch.Tensor) else torch.from_numpy(np.array(to_play, np.int32).reshape(-1))).to(torch.int32).contiguous()
                assert not h_mask.is_cuda and (h_noise is None or not h_noise.is_cuda), "host observation batch needs host mask / noise"
                self._keep_host = (h_obs, h_mask, h_noise, h_tp)
            else:
                d_obs = obs.contiguous() if u8 else obs.to(torch.float32).contiguous()
                mask_t = action_mask if isinstance(action_mask, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(action_mask))
                bufs["mask"].copy_(mask_t.to(torch.uint8), non_blocking=True)
                d_noise = None
                if noises is not None:
                    nz = noises if isinstance(noises, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(noises, dtype=np.float32))
                    bufs["noise"].copy_(nz, non_blocking=True)
                    d_noise = bufs["noise"]
                d_tp = None
                if to_play is not None:
                    tp = to_play if isinstance(to_play, torch.Tensor) else torch.from_numpy(np.array(to_play, np.int32).reshape(-1))
                    bufs["to_play"].copy_(tp.to(torch.int32), non_blocking=True)
                    d_tp = bufs["to_play"]
            tree = mz_tree.acquire_tree(dev, B, A, S)
            try:
                tree.set_params(*self.mcts._params())
                cabi.check(tree.lib.lz_tree_set_ez(tree.h, *self._tree_mode), "lz_tree_set_ez")
                q = tree.search_for(self.model, S, self._tree_mode if self._tree_mode[0] else ())
                s = cabi.stream_ptr()
                if host_path:
                    fn = tree.lib.lz_search_collect_host_u8 if u8 else tree.lib.lz_search_collect_host
                    cabi.check(fn(q, h_obs.data_ptr(), h_mask.data_ptr(), cabi.ptr(h_noise),
                                  float(self.cfg.root_noise_weight), cabi.ptr(h_tp), int(det),
                                  int(self.h2d_chunks), bufs["pred_value"].data_ptr(),
                                  bufs["logits"].data_ptr(), s), "lz_search_collect_host")
                else:
                    fn = tree.lib.lz_search_collect_u8 if u8 else tree.lib.lz_search_collect
                    cabi.check(fn(q, d_obs.data_ptr(), bufs["mask"].data_ptr(), cabi.ptr(d_noise),
                                  float(self.cfg.root_noise_weight), cabi.ptr(d_tp), int(det),
                                  bufs["pred_value"].data_ptr(), bufs["logits"].data_ptr(), s),
                               "lz_search_collect")
                cabi.check(tree.lib.lz_tree_results(tree.h, tree.visits.data_ptr(), tree.values.data_ptr(),
                                                    tree.nlegal.data_ptr(), None, s), "lz_tree_results")
                self.last_num_kernels = tree.lib.lz_search_num_kernels(q)
                if select is not None:
                    cabi.check(tree.lib.lz_tree_select_action(tree.h, float(select[0]), int(bool(select[1])), int(select[2]) & (2 ** 64 - 1),
                                                              bufs["action"].data_ptr(), bufs["action_pos"].data_ptr(),
                                                              bufs["entropy"].data_ptr(), s), "lz_tree_select_action")
                if not read_back:
                    dev_out = dict(visits=tree.visits.clone(), values=tree.values.clone(), nlegal=tree.nlegal.clone(),
                                   pred_value=bufs["pred_value"], policy_logits=bufs["logits"])
                    if select is not None:      # the device-side select_action results stay on the device too
                        dev_out.update(action=bufs["action"].clone(), entropy=bufs["entropy"].clone())
                    return dev_out
                bufs["h_visits"].copy_(tree.visits, non_blocking=True)
                bufs["h_values"].copy_(tree.values, non_blocking=True)
                bufs["h_nlegal"].copy_(tree.nlegal, non_blocking=True)
                bufs["h_pred"].copy_(bufs["pred_value"], non_blocking=True)
                bufs["h_logits"].copy_(bufs["logits"], non_blocking=True)
                if select is not None:
                    bufs["h_action"].copy_(bufs["action"], non_blocking=True)
                    bufs["h_entropy"].copy_(bufs["entropy"], non_blocking=True)
                torch.cuda.current_stream().synchronize()
            finally:
                tree.busy = False
        out = dict(visits=bufs["h_visits"], values=bufs["h_values"], nlegal=bufs["h_nlegal"],
                   pred_value=bufs["h_pred"], policy_logits=bufs["h_logits"])
        if select is not None:
            out.update(action=bufs["h_action"], entropy=bufs["h_entropy"])
        return out

    # ---- reference-shaped API --------------------------------------------------------------------
    def forward_collect(self, data: torch.Tensor, action_mask, temperature: float = 1, to_play=(-1,),
                        epsilon: float = 0.25, ready_env_id=None, device_select_action: bool = False, seed: int = 0,
                        **kwargs) -> Dict[int, dict]:
        """policy/muzero.py:705-829 (collect_with_pure_policy=False, no eps-greedy).  device_select_action=True draws the
        actions on the GPU (lz_tree_select_action, keyed by `seed`) instead of np.random.choice on the host."""
        B = data.shape[0]
        if ready_env_id is None:
            ready_env_id = np.arange(B)
        action_mask = np.asarray(action_mask)
        A = action_mask.shape[1]
        alpha = float(self.cfg.root_dirichlet_alpha)
        noises = np.zeros((B, A), np.float32)
        for j in range(B):                                   # policy/muzero.py:763-766
            n = int(action_mask[j].sum())
            noises[j, :n] = np.random.dirichlet([alpha] * n).astype(np.float32)
        tp = np.broadcast_to(np.asarray(to_play, np.int32).reshape(-1), (B,)) if np.size(to_play) in (1, B) else to_play
        r = self.search_batch(data, action_mask, noises, tp, deterministic=self.mcts.deterministic,
                              select=(temperature, False, seed) if device_select_action else None)
        return self._format(r, action_mask, ready_env_id, temperature, deterministic_action=False)

    def forward_eval(self, data: torch.Tensor, action_mask, to_play=(-1,), ready_env_id=None, **kwargs):
        """policy/muzero.py:872-956: no noise, arg-max action."""
        B = data.shape[0]
        if ready_env_id is None:
            ready_env_id = np.arange(B)
        action_mask = np.asarray(action_mask)
        tp = np.broadcast_to(np.asarray(to_play, np.int32).reshape(-1), (B,)) if np.size(to_play) in (1, B) else to_play
        r = self.search_batch(data, action_mask, None, tp, deterministic=self.mcts.deterministic)
        return self._format(r, action_mask, ready_env_id, 1, deterministic_action=True)

    def _format(self, r, action_mask, ready_env_id, temperature, deterministic_action) -> Dict[int, dict]:
        visits, nl = r["visits"].numpy(), r["nlegal"].numpy()
        values, pred, logits = r["values"].numpy(), r["pred_value"].numpy(), r["policy_logits"].numpy()
        output = {}
        for i, env_id in enumerate(ready_env_id):
            distributions = visits[i, :nl[i]].tolist()
            if "action" in r:                                              # chosen on the device
                action, ent = int(r["action"][i]), float(r["entropy"][i])
            else:
                pos, ent = select_action(distributions, temperature=temperature, deterministic=deterministic_action)
                action = np.where(action_mask[i] == 1.0)[0][pos]            # policy/muzero.py:800
            output[env_id] = {
                'action': action,
                'visit_count_distributions': distributions,
                'visit_count_distribution_entropy': ent,
                'searched_value': float(values[i]),
                'predicted_value': float(pred[i]),
                'predicted_policy_logits': logits[i].tolist(),
            }
        return output


class EfficientZeroCollectPolicy(MuZeroCollectPolicy):
    """The same for ``EfficientZeroPolicy._forward_collect`` / ``_forward_eval`` (lzero/policy/efficientzero.py:539-640,
    690-760): value-prefix trees, the reward hidden state starts as zeros after ``initial_inference`` (:580-590) and is reset
    every ``lstm_horizon_len`` steps of search depth.  Same output dict."""

    def __init__(self, model: EfficientZeroModel, cfg: Optional[dict] = None):
        super().__init__(model, cfg)
        self.mcts = EfficientZeroMCTSCtree(cfg or {})
        self.cfg = self.mcts._cfg
        self._tree_mode = (1, int(self.cfg.lstm_horizon_len))


class GumbelMuZeroCollectPolicy:
    """``GumbelMuZeroPolicy._forward_collect`` / ``_forward_eval`` (lzero/policy/gumbel_muzero.py:520-607, 619-705): initial
    inference, roots prepared with the predicted values, the Gumbel search (one CUDA graph with a ``lightzero_b200`` model) and
    the per-environment output dict.  Everything stays on the device until ONE read-back per step: the action (arg-max of
    the improved policy with illegal entries 0, :591-592, computed by ``lz_tree_results_gumbel``), the visit counts, the
    visit-count entropy (``lz_tree_select_action``), the searched value, the completed values (0 off the legal list), the
    improved policy, the predicted value and the policy logits."""

    def __init__(self, model, cfg: Optional[dict] = None):
        from .mcts_ctree import GumbelMuZeroMCTSCtree
        self.model = model
        self.mcts = GumbelMuZeroMCTSCtree(cfg or {})
        self.cfg = self.mcts._cfg
        self.device = model.device

    def _step(self, data, action_mask, noises, to_play, temperature):
        from . import gmz_tree
        action_mask = np.asarray(action_mask)
        B, A = action_mask.shape
        dev = self.device
        self.mcts._make_inverse_transforms(dev)
        with torch.no_grad(), torch.cuda.device(dev):
            out = self.model.initial_inference(data.to(dev, non_blocking=True))
            pred = self.mcts._inv(out.value).reshape(-1).contiguous()              # gumbel_muzero.py:546 (inverse transform)
            roots = gmz_tree.Roots(B, action_mask.astype(np.uint8))
            if noises is None:
                roots.prepare_no_noise(None, pred, out.policy_logits, to_play)
            else:
                roots.prepare(float(self.cfg.root_noise_weight), noises, None, pred, out.policy_logits, to_play)
            self.mcts.search(roots, self.model, out.latent_state, to_play)
            visits, nlegal = roots.get_distributions_tensor()
            values = roots.get_values_tensor()
            cv, pol, act = roots.results_tensor(float(self.cfg.discount_factor), A)
            _, _, ent = roots.select_action_tensor(temperature, deterministic=noises is None)
            mask = torch.from_numpy(action_mask != 0).to(dev)
            cv = torch.where(mask, cv, torch.zeros_like(cv))                        # :593
            flat = torch.cat([act.float(), nlegal.float(), ent, values, pred, visits.float().reshape(-1), cv.reshape(-1),
                              pol.reshape(-1), out.policy_logits.float().reshape(-1)]).cpu().numpy()   # the one read-back
            roots.clear()
        cols = [B, B, B, B, B, B * A, B * A, B * A, B * A]
        parts = np.split(flat, np.cumsum(cols)[:-1])
        act, nl, ent, values, pred = parts[:5]
        visits, cv, pol, logits = (p.reshape(B, A) for p in parts[5:])
        return act.astype(np.int64), nl.astype(np.int64), ent, values, pred, visits.astype(np.int64), cv, pol, logits

    def forward_collect(self, data: torch.Tensor, action_mask, temperature: float = 1, to_play=(-1,), ready_env_id=None,
                        **kwargs) -> Dict[int, dict]:
        """gumbel_muzero.py:520-607: Dirichlet noise over the legal actions (:553-556) drawn with np.random as the reference."""
        action_mask = np.asarray(action_mask)
        B, A = action_mask.shape
        if ready_env_id is None:
            ready_env_id = np.arange(B)
        alpha = float(self.cfg.root_dirichlet_alpha)
        noises = np.zeros((B, A), np.float32)
        for j in range(B):
            n = int(action_mask[j].sum())
            noises[j, :n] = np.random.dirichlet([alpha] * n).astype(np.float32)
        tp = np.broadcast_to(np.asarray(to_play, np.int32).reshape(-1), (B,)) if np.size(to_play) in (1, B) else np.asarray(to_play)
        act, nl, ent, values, pred, visits, cv, pol, logits = self._step(data, action_mask, noises, tp.tolist(), temperature)
        output = {}
        for i, env_id in enumerate(ready_env_id):
            output[env_id] = {
                'action': int(act[i]),
                'visit_count_distributions': visits[i, :nl[i]].tolist(),
                'visit_count_distribution_entropy': float(ent[i]),
                'searched_value': float(values[i]),
                'roots_completed_value': cv[i],
                'improved_policy_probs': pol[i],
                'predicted_value': float(pred[i]),
                'predicted_policy_logits': logits[i].tolist(),
            }
        return output

    def forward_eval(self, data: torch.Tensor, action_mask, to_play=(-1,), ready_env_id=None, **kwargs) -> Dict[int, dict]:
        """gumbel_muzero.py:619-705: no noise, the same action rule."""
        action_mask = np.asarray(action_mask)
        B = action_mask.shape[0]
        if ready_env_id is None:
            ready_env_id = np.arange(B)
        tp = np.broadcast_to(np.asarray(to_play, np.int32).reshape(-1), (B,)) if np.size(to_play) in (1, B) else np.asarray(to_play)
        act, nl, ent, values, pred, visits, cv, pol, logits = self._step(data, action_mask, None, tp.tolist(), 1.0)
        return {env_id: {
            'action': int(act[i]),
            'visit_count_distributions': visits[i, :nl[i]].tolist(),
            'visit_count_distribution_entropy': float(ent[i]),
            'searched_value': float(values[i]),
            'predicted_value': float(pred[i]),
            'predicted_policy_logits': logits[i].tolist(),
        } for i, env_id in enumerate(ready_env_id)}
