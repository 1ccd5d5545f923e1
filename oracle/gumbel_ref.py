"""oracle/gumbel_ref.py -- the Gumbel MuZero reference: builds the UNMODIFIED reference tree
lzero/mcts/ctree/ctree_gumbel_muzero (gmz_tree.pyx + .pxd, lib/cnode.cpp, cnode.h, common_lib) into oracle/_ref/gmz_tree*.so,
and restates ``GumbelMuZeroMCTSCtree.search`` (lzero/mcts/tree_search/mcts_ctree.py:1076-1174) on it.

TEST INFRASTRUCTURE ONLY, like the rest of oracle/: the product package never imports it.  The build follows the recipe of
oracle/build_ref.py (Cython in place, generated C++ to a temp dir, g++ -std=c++11 -O2 -DNDEBUG, the same include-path quirk).
The Gumbel tree's search path never calls rand() (cbatch_traverse reseeds srand, but cselect_root_child /
cselect_interior_child are arg-max scans and the Gumbel draw is a fixed std::mt19937(0)), so no rand() shim is linked.
"""
import copy
import os
import subprocess
import sys
import sysconfig
import tempfile

import numpy as np
import torch

from oracle import build_ref
from oracle.search_ref import SearchRef

NAME, SUBDIR = "gmz_tree", "ctree_gumbel_muzero"


def module_path() -> str:
    return build_ref.ref_module_path(NAME)


def build(force: bool = False) -> str:
    """Returns the path of the built module, or '' if the reference tree is absent."""
    target = module_path()
    if os.path.exists(target) and not force:
        return target
    src_dir = os.path.join(build_ref.CTREE, SUBDIR)
    if not os.path.isdir(src_dir):
        return ""
    import numpy
    os.makedirs(os.path.dirname(target), exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        gen_cpp = os.path.join(tmp, NAME + ".cpp")
        subprocess.check_call([sys.executable, "-m", "cython", "--cplus", "-3", "-I", src_dir,
                               os.path.join(src_dir, NAME + ".pyx"), "-o", gen_cpp])
        inc = sysconfig.get_paths()["include"]
        subprocess.check_call(["g++", "-std=c++11", "-O2", "-DNDEBUG", "-fPIC", "-shared", "-w",
                               "-I", inc, "-I", numpy.get_include(), "-I", src_dir, "-I", os.path.join(src_dir, "lib"),
                               "-I", build_ref.CTREE, gen_cpp, "-o", target])
    return target


def load():
    """The compiled reference module, or None when it was not built."""
    path = module_path()
    if not os.path.exists(path):
        return None
    d = os.path.dirname(path)
    if d not in sys.path:
        sys.path.insert(0, d)
    import gmz_tree
    return gmz_tree


class GumbelSearchRef(SearchRef):
    """GumbelMuZeroMCTSCtree.search (mcts_ctree.py:1076-1174) on the compiled gmz_tree, with the recorder / replay hooks of
    SearchRef.search.  Roots come from tree.Roots(n, legal) and are prepared by the caller with values (gmz_tree.pyx:36-40)."""

    def __init__(self, tree_module, num_simulations=50, max_num_considered_actions=4, **kw):
        super().__init__(tree_module, num_simulations=num_simulations, **kw)
        self.max_num_considered_actions = max_num_considered_actions

    def search(self, roots, model, latent_state_roots, to_play_batch, recorder=None, replay=None):
        tree = self.tree
        with torch.no_grad():
            if model is not None:
                model.eval()
            batch_size = roots.num
            latent_pool = [latent_state_roots]
            mm = tree.MinMaxStatsList(batch_size)
            mm.set_delta(self.value_delta_max)
            for simulation_index in range(self.num_simulations):
                results = tree.ResultsWrapper(batch_size)
                tp_arg = to_play_batch if self.env_type == "not_board_games" else copy.deepcopy(to_play_batch)
                ix_l, iy_l, last_actions, virtual_to_play = tree.batch_traverse(
                    roots, self.num_simulations, self.max_num_considered_actions, self.discount_factor, results, list(tp_arg))
                if replay is not None:
                    rec = replay[simulation_index]
                    reward_batch, value_batch, policy_logits_batch = rec["reward"], rec["value"], rec["policy"]
                else:
                    latent_states = torch.from_numpy(np.asarray([latent_pool[ix][iy] for ix, iy in zip(ix_l, iy_l)]))
                    out = model.recurrent_inference(latent_states, torch.from_numpy(np.asarray(last_actions)).long())
                    latent_pool.append(out.latent_state.detach().cpu().numpy())
                    reward_batch = self.reward_inv(out.reward).detach().cpu().numpy().reshape(-1).tolist()
                    value_batch = self.value_inv(out.value).detach().cpu().numpy().reshape(-1).tolist()
                    policy_logits_batch = out.policy_logits.detach().cpu().numpy().tolist()
                if recorder is not None:
                    recorder.append(dict(ix=list(ix_l), iy=list(iy_l), last_action=list(last_actions),
                                         search_len=list(results.get_search_len()),
                                         reward=list(reward_batch), value=list(value_batch),
                                         policy=[list(p) for p in policy_logits_batch]))
                tree.batch_back_propagate(simulation_index + 1, self.discount_factor, reward_batch, value_batch,
                                          policy_logits_batch, mm, results, virtual_to_play)
        return latent_pool


def gumbel_search_step_ref(search: GumbelSearchRef, model, obs, legal, noises, to_play, noise_weight=0.25):
    """initial_inference -> Roots.prepare(noise, values) -> search on the CPU oracle pipeline; returns the root statistics."""
    with torch.no_grad():
        model.eval()
        out = model.initial_inference(obs)
        values = search.value_inv(out.value).reshape(-1).cpu().numpy()
    B = obs.shape[0]
    roots = search.tree.Roots(B, legal)
    roots.prepare(noise_weight, noises, [0.] * B, values.tolist(), out.policy_logits.cpu().numpy().tolist(), list(to_play))
    search.search(roots, model, out.latent_state.cpu().numpy(), list(to_play))
    return dict(distributions=roots.get_distributions(), values=roots.get_values(), pred_values=values,
                policy_logits=out.policy_logits.cpu().numpy(), latent=out.latent_state)


if __name__ == "__main__":
    p = build(force="--force" in sys.argv)
    print(p if p else "reference tree not present; nothing built")
