"""Golden fixtures for the Gumbel MuZero tree, written by RUNNING THE COMPILED, UNMODIFIED REFERENCE
(oracle/_ref/gmz_tree, built by oracle/gumbel_ref.py from lzero/mcts/ctree/ctree_gumbel_muzero).

    python tests/golden/make_gumbel_golden.py

Each fixture gumbel_<name>.npz is a replay-mode trace: every input the tree consumes (legal lists, root logits / values /
rewards, noise, per-simulation reward / value / policy-logit batches) and everything it produces: per simulation
(ix, iy, last_action, search_len, virtual_to_play), and at the end the visit distributions, root-value bits, best-action
trajectories, children-value bits and improved-policy bits.  The Gumbel search draws no random numbers, so no shim is needed.

The helpers (make_inputs, run_reference, run_cuda) are shared with tests/test_gpu_gumbel.py and tests/test_gumbel_cpu.py.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DISCOUNT, NOISE_W = 0.997, 0.25

CASES = [
    # name,              B,  A,  S,  m, masks, noise, two_player, scale, seed
    ("atari_a18_m4",     32, 18, 50,  4, 0, 1, 0, 1.0, 11),
    ("atari_a18_mask",   32, 18, 50, 18, 1, 1, 0, 3.0, 12),
    ("deep_s200",         8, 18, 200, 4, 1, 0, 0, 0.3, 13),
    ("wide_a40",          6, 40, 40, 16, 0, 1, 0, 3.0, 14),
    ("masked_2p_a9",     16,  9, 30, 16, 2, 1, 1, 1.0, 15),
    ("cartpole_a2",       8,  2, 25,  2, 0, 1, 0, 1.0, 16),
    ("degenerate_a1",     3,  1,  5,  1, 0, 0, 0, 1.0, 17),
]


def make_inputs(B, A, S, masks, noise, two_player, scale, seed):
    """masks: 0 = all legal, 1 = ~60 % legal, 2 = at most 3 legal (fewer than m: the all -inf root branch)."""
    rng = np.random.default_rng(seed)
    legal = []
    for _ in range(B):
        if masks == 0:
            mk = np.ones(A, bool)
        else:
            mk = rng.random(A) < (0.6 if masks == 1 else 0.25)
            if masks == 2 and mk.sum() > 3:
                mk[np.nonzero(mk)[0][3:]] = False
            mk[rng.integers(A)] = True
        legal.append(np.nonzero(mk)[0].tolist())
    f32 = np.float32
    inp = dict(B=B, A=A, S=S, scale=scale, legal=legal,
               logits=(rng.standard_normal((B, A)) * scale).astype(f32),
               values=(rng.standard_normal(B) * scale).astype(f32),
               rewards=(rng.standard_normal(B) * scale * 0.1).astype(f32),
               to_play=(rng.integers(1, 3, size=B) if two_player else np.full(B, -1)).astype(np.int32),
               noise=None,
               rew=(rng.standard_normal((S, B)) * scale).astype(f32),
               val=(rng.standard_normal((S, B)) * scale).astype(f32),
               pol=(rng.standard_normal((S, B, A)) * scale).astype(f32))
    if noise:
        inp["noise"] = [rng.dirichlet([0.3] * len(l)).astype(f32).tolist() for l in legal]
    return inp


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def run_reference(gmz, inp, m, discount=DISCOUNT):
    """GumbelMuZeroMCTSCtree.search's tree calls (mcts_ctree.py:1076-1174) on the compiled reference, fed recorded outputs."""
    B, A, S = inp["B"], inp["A"], inp["S"]
    roots = gmz.Roots(B, inp["legal"])
    tp = inp["to_play"].tolist()
    if inp["noise"] is not None:
        roots.prepare(NOISE_W, inp["noise"], inp["rewards"].tolist(), inp["values"].tolist(), inp["logits"].tolist(), tp)
    else:
        roots.prepare_no_noise(inp["rewards"].tolist(), inp["values"].tolist(), inp["logits"].tolist(), tp)
    mm = gmz.MinMaxStatsList(B)
    mm.set_delta(0.01)
    trace = {k: np.zeros((S, B), np.int32) for k in ("ix", "iy", "last_action", "vtp", "search_len")}
    for s in range(S):
        res = gmz.ResultsWrapper(B)
        ix, iy, la, vtp = gmz.batch_traverse(roots, S, m, discount, res, list(tp))
        trace["ix"][s], trace["iy"][s], trace["last_action"][s], trace["vtp"][s] = ix, iy, la, vtp
        trace["search_len"][s] = res.get_search_len()
        gmz.batch_back_propagate(s + 1, discount, inp["rew"][s].tolist(), inp["val"][s].tolist(), inp["pol"][s].tolist(), mm, res, vtp)
    return _final(roots, trace, discount, A)


def _final(roots, trace, discount, A):
    dist = roots.get_distributions()
    traj = roots.get_trajectories()
    out = dict(trace)
    out["dist"] = dist
    out["value_bits"] = _bits(roots.get_values())
    out["traj"] = traj
    out["children_value_bits"] = _bits(roots.get_children_values(discount, A))
    out["policy_bits"] = _bits(roots.get_policies(discount, A))
    return out


def run_cuda(inp, m, discount=DISCOUNT, tensors=False):
    """The same calls on lightzero_b200.gmz_tree; tensors=True passes every input as a CUDA tensor."""
    import torch
    from lightzero_b200 import gmz_tree as gmz
    B, A, S = inp["B"], inp["A"], inp["S"]

    def arg(x):
        if not tensors or x is None:
            return x.tolist() if isinstance(x, np.ndarray) else x
        if isinstance(x, list):      # noise rows in legal order -> [B, A] zero padded
            arr = np.zeros((B, A), np.float32)
            for i, r in enumerate(x):
                arr[i, :len(r)] = r
            x = arr
        return torch.from_numpy(np.ascontiguousarray(x)).cuda()
    roots = gmz.Roots(B, inp["legal"])
    tp = arg(inp["to_play"])
    if inp["noise"] is not None:
        roots.prepare(NOISE_W, arg(inp["noise"]), arg(inp["rewards"]), arg(inp["values"]), arg(inp["logits"]), tp)
    else:
        roots.prepare_no_noise(arg(inp["rewards"]), arg(inp["values"]), arg(inp["logits"]), tp)
    mm = gmz.MinMaxStatsList(B)
    mm.set_delta(0.01)
    trace = {k: np.zeros((S, B), np.int32) for k in ("ix", "iy", "last_action", "vtp", "search_len")}
    for s in range(S):
        res = gmz.ResultsWrapper(B)
        ix, iy, la, vtp = gmz.batch_traverse(roots, S, m, discount, res, inp["to_play"].tolist())
        trace["ix"][s], trace["iy"][s], trace["last_action"][s], trace["vtp"][s] = ix, iy, la, vtp
        trace["search_len"][s] = res.get_search_len()
        gmz.batch_back_propagate(s + 1, discount, arg(inp["rew"][s]), arg(inp["val"][s]), arg(inp["pol"][s]), mm, res, vtp)
    out = _final(roots, trace, discount, A)
    roots.clear()
    return out


def load_reference():
    """The compiled reference module, or None when oracle/_ref/gmz_tree was not built."""
    from oracle import gumbel_ref
    return gumbel_ref.load()


def save_fixture(path, inp, m, out):
    B, A = inp["B"], inp["A"]
    legal = np.full((B, A), -1, np.int32)
    for i, l in enumerate(inp["legal"]):
        legal[i, :len(l)] = l
    noise = np.zeros((B, A), np.float32)
    if inp["noise"] is not None:
        for i, r in enumerate(inp["noise"]):
            noise[i, :len(r)] = r
    S = inp["S"]
    traj = np.full((B, S + 1), -1, np.int32)
    for i, t in enumerate(out["traj"]):
        traj[i, :len(t)] = t
    dist = np.full((B, A), -1, np.int32)
    for i, d in enumerate(out["dist"]):
        dist[i, :len(d)] = d
    np.savez_compressed(path, B=B, A=A, S=S, m=m, discount=np.float32(DISCOUNT), has_noise=int(inp["noise"] is not None),
                        legal=legal, logits=inp["logits"], values=inp["values"], rewards=inp["rewards"], to_play=inp["to_play"],
                        noise=noise, rew=inp["rew"], val=inp["val"], pol=inp["pol"],
                        ix=out["ix"], iy=out["iy"], last_action=out["last_action"], vtp=out["vtp"], search_len=out["search_len"],
                        dist=dist, value_bits=out["value_bits"], traj=traj, children_value_bits=out["children_value_bits"],
                        policy_bits=out["policy_bits"])


def load_fixture(path):
    z = np.load(path)
    B, A = int(z["B"]), int(z["A"])
    legal = [[int(a) for a in row if a >= 0] for row in z["legal"]]
    noise = None
    if int(z["has_noise"]):
        noise = [z["noise"][i, :len(l)].tolist() for i, l in enumerate(legal)]
    inp = dict(B=B, A=A, S=int(z["S"]), legal=legal, logits=z["logits"], values=z["values"], rewards=z["rewards"],
               to_play=z["to_play"], noise=noise, rew=z["rew"], val=z["val"], pol=z["pol"])
    exp = {k: z[k] for k in ("ix", "iy", "last_action", "vtp", "search_len", "value_bits", "children_value_bits", "policy_bits")}
    exp["dist"] = [[int(v) for v in row if v >= 0] for row in z["dist"]]
    exp["traj"] = [[int(v) for v in row if v >= 0] for row in z["traj"]]
    return inp, int(z["m"]), exp


def main():
    gmz = load_reference()
    assert gmz is not None, "build oracle/_ref/gmz_tree first (python -m oracle.gumbel_ref)"
    for name, B, A, S, m, masks, noise, two_player, scale, seed in CASES:
        inp = make_inputs(B, A, S, masks, noise, two_player, scale, seed)
        out = run_reference(gmz, inp, m)
        path = os.path.join(HERE, f"gumbel_{name}.npz")
        save_fixture(path, inp, m, out)
        print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
