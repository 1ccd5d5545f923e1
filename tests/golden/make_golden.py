"""Generate the committed golden fixtures for the MuZero and EfficientZero ctree paths by RUNNING THE COMPILED,
UNMODIFIED REFERENCE (oracle/_ref/mz_tree and ez_tree, built from /root/reference by oracle/build_ref.py; ez_tree
is linked with oracle/rand_shim.c so that its rand()-based tie-break is reproducible).

Run in the build container (the GPU box has no /root/reference; it uses the committed .npz files):
    python tests/golden/make_golden.py

Each fixture is a replay-mode trace: all inputs the tree consumes (legal lists, root logits,
Dirichlet noise, per-simulation reward / value / policy-logit batches) and everything it produces
(per-simulation (ix, iy, last_action, search_len, virtual_to_play), final visit distributions,
root values as raw fp32 bits, best-action trajectories).  deterministic=True (SURVEY.md s.0 fact 2).
"""
import copy
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))

CASES = [
    # name,            B,  A,  S,  masks, noise, two_player, scale, seed
    ("survey_b4a6",     4,  6, 10, 0, 0, 0, 1.0, 0),   # SURVEY.md 8c session vector (same draws)
    ("atari_a6",       32,  6, 50, 0, 1, 0, 1.0, 1),
    ("atari_a18",      32, 18, 50, 0, 1, 0, 1.0, 2),
    ("atari_a18_mask", 32, 18, 50, 1, 1, 0, 2.0, 3),
    ("deep_s200",       8, 18, 200, 0, 1, 0, 0.5, 4),
    ("board_2p_a9",    16,  9, 40, 1, 1, 1, 1.0, 5),
    ("wide_a40",        6, 40, 60, 1, 0, 0, 3.0, 6),
    ("cartpole_a2",     8,  2, 25, 0, 1, 0, 1.0, 7),
]
PB_C_BASE, PB_C_INIT, DISCOUNT, DELTA, NOISE_W = 19652, 1.25, 0.997, 0.01, 0.25


def make_case(mz, B, A, S, masks, noise, two_player, scale, seed):
    rng = np.random.default_rng(seed)
    if masks:
        legal = []
        for _ in range(B):
            m = rng.random(A) < 0.6
            if not m.any():
                m[rng.integers(A)] = True
            legal.append(np.nonzero(m)[0].tolist())
    else:
        legal = [list(range(A)) for _ in range(B)]
    pol = (rng.standard_normal((B, A)) * scale).astype(np.float32)
    to_play = rng.integers(1, 3, size=B).astype(np.int32) if two_player else np.full(B, -1, np.int32)
    roots = mz.Roots(B, legal)
    noises = np.zeros((B, A), np.float32)
    if noise:
        nz = []
        for b, l in enumerate(legal):
            d = rng.dirichlet([0.3] * len(l)).astype(np.float32)
            noises[b, :len(l)] = d
            nz.append(d.tolist())
        roots.prepare(NOISE_W, nz, [0.] * B, pol.tolist(), to_play.tolist())
    else:
        roots.prepare_no_noise([0.] * B, pol.tolist(), to_play.tolist())
    mm = mz.MinMaxStatsList(B)
    mm.set_delta(DELTA)
    rew = np.zeros((S, B), np.float32); val = np.zeros((S, B), np.float32)
    pols = np.zeros((S, B, A), np.float32)
    ix = np.zeros((S, B), np.int32); iy = np.zeros((S, B), np.int32)
    la = np.zeros((S, B), np.int32); sl = np.zeros((S, B), np.int32); vtp = np.zeros((S, B), np.int32)
    for s in range(S):
        res = mz.ResultsWrapper(B)
        a, b_, c, d = mz.batch_traverse(roots, PB_C_BASE, PB_C_INIT, DISCOUNT, mm, res,
                                        copy.deepcopy(to_play.tolist()), True)
        ix[s], iy[s], la[s], vtp[s] = a, b_, c, d
        sl[s] = res.get_search_len()
        # draw order matches SURVEY.md 8c: r, v, p
        rew[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        val[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        pols[s] = (rng.standard_normal((B, A)) * scale).astype(np.float32)
        mz.batch_backpropagate(s + 1, DISCOUNT, rew[s].tolist(), val[s].tolist(), pols[s].tolist(), mm, res, d)
    dist = np.full((B, A), -1, np.int32)
    for b, dd in enumerate(roots.get_distributions()):
        dist[b, :len(dd)] = dd
    values = np.asarray(roots.get_values(), np.float32)
    traj = np.full((B, S + 1), -1, np.int32)
    for b, t in enumerate(roots.get_trajectories()):
        traj[b, :len(t)] = t
    legal_arr = np.full((B, A), -1, np.int32)
    nlegal = np.zeros(B, np.int32)
    for b, l in enumerate(legal):
        legal_arr[b, :len(l)] = l
        nlegal[b] = len(l)
    return dict(B=B, A=A, S=S, use_noise=noise, legal=legal_arr, nlegal=nlegal, root_logits=pol,
                noises=noises, to_play=to_play, rewards=rew, values_in=val, policies=pols,
                ix=ix, iy=iy, last_action=la, search_len=sl, virtual_to_play=vtp,
                distributions=dist, root_values_bits=values.view(np.uint32), trajectories=traj,
                pb_c_base=PB_C_BASE, pb_c_init=np.float32(PB_C_INIT), discount=np.float32(DISCOUNT),
                delta=np.float32(DELTA), noise_w=np.float32(NOISE_W))


EZ_CASES = [
    # name,             B,  A,  S,  masks, noise, two_player, scale, seed, lstm_horizon_len
    ("ez_atari_a6",     32,  6, 50, 0, 1, 0, 1.0, 11, 5),
    ("ez_atari_a18",    32, 18, 50, 1, 1, 0, 2.0, 12, 5),
    ("ez_deep_s120",     8, 18, 120, 0, 1, 0, 0.5, 13, 3),
    ("ez_board_2p_a9",  16,  9, 40, 1, 1, 1, 1.0, 14, 4),
]


def make_case_ez(ez, B, A, S, masks, noise, two_player, scale, seed, horizon):
    """EfficientZero tree (oracle/_ref/ez_tree = unmodified ctree_efficientzero + rand()==0 shim): the driver protocol of
    mcts_ctree.py:782-876 -- value prefixes instead of rewards, is_reset = (search_len % lstm_horizon_len == 0)."""
    rng = np.random.default_rng(seed)
    if masks:
        legal = []
        for _ in range(B):
            m = rng.random(A) < 0.6
            if not m.any():
                m[rng.integers(A)] = True
            legal.append(np.nonzero(m)[0].tolist())
    else:
        legal = [list(range(A)) for _ in range(B)]
    pol = (rng.standard_normal((B, A)) * scale).astype(np.float32)
    to_play = rng.integers(1, 3, size=B).astype(np.int32) if two_player else np.full(B, -1, np.int32)
    roots = ez.Roots(B, legal)
    noises = np.zeros((B, A), np.float32)
    if noise:
        nz = []
        for b, l in enumerate(legal):
            d = rng.dirichlet([0.3] * len(l)).astype(np.float32)
            noises[b, :len(l)] = d
            nz.append(d.tolist())
        roots.prepare(NOISE_W, nz, [0.] * B, pol.tolist(), to_play.tolist())
    else:
        roots.prepare_no_noise([0.] * B, pol.tolist(), to_play.tolist())
    mm = ez.MinMaxStatsList(B)
    mm.set_delta(DELTA)
    vp = np.zeros((S, B), np.float32); val = np.zeros((S, B), np.float32)
    pols = np.zeros((S, B, A), np.float32)
    ix = np.zeros((S, B), np.int32); iy = np.zeros((S, B), np.int32)
    la = np.zeros((S, B), np.int32); sl = np.zeros((S, B), np.int32); vtp = np.zeros((S, B), np.int32)
    rs = np.zeros((S, B), np.int32)
    for s in range(S):
        res = ez.ResultsWrapper(B)
        a, b_, c, d = ez.batch_traverse(roots, PB_C_BASE, PB_C_INIT, DISCOUNT, mm, res, copy.deepcopy(to_play.tolist()))
        ix[s], iy[s], la[s], vtp[s] = a, b_, c, d
        sl[s] = res.get_search_len()
        vp[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        val[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        pols[s] = (rng.standard_normal((B, A)) * scale).astype(np.float32)
        rs[s] = (sl[s] % horizon == 0).astype(np.int32)
        ez.batch_backpropagate(s + 1, DISCOUNT, vp[s].tolist(), val[s].tolist(), pols[s].tolist(), mm, res,
                               rs[s].tolist(), d)
    dist = np.full((B, A), -1, np.int32)
    for b, dd in enumerate(roots.get_distributions()):
        dist[b, :len(dd)] = dd
    values = np.asarray(roots.get_values(), np.float32)
    traj = np.full((B, S + 1), -1, np.int32)
    for b, t in enumerate(roots.get_trajectories()):
        traj[b, :len(t)] = t
    legal_arr = np.full((B, A), -1, np.int32)
    nlegal = np.zeros(B, np.int32)
    for b, l in enumerate(legal):
        legal_arr[b, :len(l)] = l
        nlegal[b] = len(l)
    return dict(B=B, A=A, S=S, use_noise=noise, legal=legal_arr, nlegal=nlegal, root_logits=pol,
                noises=noises, to_play=to_play, rewards=vp, values_in=val, policies=pols, is_reset=rs,
                ix=ix, iy=iy, last_action=la, search_len=sl, virtual_to_play=vtp,
                distributions=dist, root_values_bits=values.view(np.uint32), trajectories=traj,
                pb_c_base=PB_C_BASE, pb_c_init=np.float32(PB_C_INIT), discount=np.float32(DISCOUNT),
                delta=np.float32(DELTA), noise_w=np.float32(NOISE_W), lstm_horizon_len=horizon)


REUSE_CASES = [
    # name,               tree,      B,  A,  S, masks, noise, two_player, scale, seed, lstm_horizon_len (EZ only)
    ("reuse_mz_a6",       "mz",     32,  6, 40, 0, 1, 0, 1.0, 21, 0),
    ("reuse_mz_a18_mask", "mz",     24, 18, 40, 1, 1, 0, 2.0, 22, 0),
    ("reuse_mz_2p_a9",    "mz",     16,  9, 30, 1, 1, 1, 1.0, 23, 0),
    ("reuse_ez_a6",       "ez",     32,  6, 40, 0, 1, 0, 1.0, 24, 3),
]


def make_case_reuse(mod, B, A, S, masks, noise, two_player, scale, seed, horizon):
    """ReZero *_with_reuse (mcts_ctree.py:370-468 / :878-1000 protocol) on the rand() == 0 builds: besides the usual trace the
    fixture stores true_action / reuse_value, the compacted network outputs of every simulation (padded to B rows, n_inferred says
    how many are real) and the -1 terminated no_inference / reuse lists the driver builds."""
    rng = np.random.default_rng(seed)
    legal = []
    for _ in range(B):
        m = rng.random(A) < 0.6 if masks else np.ones(A, bool)
        if not m.any():
            m[rng.integers(A)] = True
        legal.append(np.nonzero(m)[0].tolist())
    pol = (rng.standard_normal((B, A)) * scale).astype(np.float32)
    to_play = rng.integers(1, 3, size=B).astype(np.int32) if two_player else np.full(B, -1, np.int32)
    true_action = np.asarray([int(l[rng.integers(len(l))]) for l in legal], np.int32)
    reuse_value = (rng.standard_normal(B) * scale).astype(np.float32)
    roots = mod.Roots(B, legal)
    noises = np.zeros((B, A), np.float32)
    if noise:
        nz = []
        for b, l in enumerate(legal):
            d = rng.dirichlet([0.3] * len(l)).astype(np.float32)
            noises[b, :len(l)] = d
            nz.append(d.tolist())
        roots.prepare(NOISE_W, nz, [0.] * B, pol.tolist(), to_play.tolist())
    else:
        roots.prepare_no_noise([0.] * B, pol.tolist(), to_play.tolist())
    mm = mod.MinMaxStatsList(B)
    mm.set_delta(DELTA)
    rew = np.zeros((S, B), np.float32); val = np.zeros((S, B), np.float32); pols = np.zeros((S, B, A), np.float32)
    ix = np.zeros((S, B), np.int32); iy = np.zeros((S, B), np.int32); la = np.zeros((S, B), np.int32)
    sl = np.zeros((S, B), np.int32); vtp = np.zeros((S, B), np.int32); rs = np.zeros((S, B), np.int32)
    n_inf = np.zeros(S, np.int32)
    no_inf = np.full((S, B + 1), -1, np.int32); reuse = np.full((S, B + 1), -1, np.int32)
    for s in range(S):
        res = mod.ResultsWrapper(B)
        a, b_, c, d = mod.batch_traverse_with_reuse(roots, PB_C_BASE, PB_C_INIT, DISCOUNT, mm, res, copy.deepcopy(to_play.tolist()),
                                                    true_action.tolist(), reuse_value.tolist())
        ix[s], iy[s], la[s], vtp[s] = a, b_, c, d
        sl[s] = res.get_search_len()
        ni, ru, n = [], [], 0
        for count, (x, y) in enumerate(zip(a, b_)):
            if x != -1:
                n += 1
            else:
                ni.append(y)
            if x == 0 and c[count] == true_action[count]:
                ru.append(count)
        n_inf[s] = n
        no_inf[s, :len(ni)] = ni
        reuse[s, :len(ru)] = ru
        rew[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        val[s] = (rng.standard_normal(B) * scale).astype(np.float32)
        pols[s] = (rng.standard_normal((B, A)) * scale).astype(np.float32)
        args = (s + 1, DISCOUNT, rew[s, :n].tolist(), val[s, :n].tolist(), pols[s, :n].tolist(), mm, res)
        if horizon:
            rs[s] = (sl[s] % horizon == 0).astype(np.int32)
            mod.batch_backpropagate_with_reuse(*args, rs[s].tolist(), d, ni + [-1], ru + [-1], reuse_value.tolist())
        else:
            mod.batch_backpropagate_with_reuse(*args, d, ni + [-1], ru + [-1], reuse_value.tolist())
    dist = np.full((B, A), -1, np.int32)
    for b, dd in enumerate(roots.get_distributions()):
        dist[b, :len(dd)] = dd
    values = np.asarray(roots.get_values(), np.float32)
    legal_arr = np.full((B, A), -1, np.int32)
    nlegal = np.zeros(B, np.int32)
    for b, l in enumerate(legal):
        legal_arr[b, :len(l)] = l
        nlegal[b] = len(l)
    return dict(B=B, A=A, S=S, use_noise=noise, legal=legal_arr, nlegal=nlegal, root_logits=pol, noises=noises, to_play=to_play,
                true_action=true_action, reuse_value=reuse_value, rewards=rew, values_in=val, policies=pols, n_inferred=n_inf,
                no_inference=no_inf, reuse_list=reuse, is_reset=rs, ix=ix, iy=iy, last_action=la, search_len=sl, virtual_to_play=vtp,
                distributions=dist, root_values_bits=values.view(np.uint32), pb_c_base=PB_C_BASE, pb_c_init=np.float32(PB_C_INIT),
                discount=np.float32(DISCOUNT), delta=np.float32(DELTA), noise_w=np.float32(NOISE_W), lstm_horizon_len=horizon)


def record_random_runs(mz, ez, mz_rand0):
    """tests/golden/ref_random_runs.json.gz: the compiled reference's results of every random run test_oracle_pin.py compares
    the C port against (RANDOM_RUNS there), each run twice to show the record is reproducible."""
    import gzip
    import json
    sys.path.insert(0, os.path.dirname(HERE))
    from test_oracle_pin import RANDOM_RUNS, random_run_cases, summarize_run
    mods = {"mz": mz, "ez": ez, "reuse_mz": mz_rand0, "reuse_ez": ez}
    rec = {}
    for tree, (run, seeds, _) in RANDOM_RUNS.items():
        for seed in seeds:
            for key, args in random_run_cases(tree, seed):
                rec[key] = summarize_run(run(mods[tree], False, *args))
                assert summarize_run(run(mods[tree], False, *args)) == rec[key], key
    with gzip.GzipFile(os.path.join(HERE, "ref_random_runs.json.gz"), "wb", compresslevel=9, mtime=0) as f:
        f.write(json.dumps(rec, sort_keys=True, separators=(",", ":")).encode())
    print("random runs recorded:", len(rec))


def main():
    import mz_tree
    for name, *args in CASES:
        case = make_case(mz_tree, *args)
        np.savez_compressed(os.path.join(HERE, f"tree_{name}.npz"), **case)
        print(name, "sum visits ok:", bool((np.where(case["distributions"] < 0, 0, case["distributions"]).sum(1) == case["S"]).all()))
    # the reference's own known-answer test (lzero/mcts/tests/test_muzero_ctree_deterministic.py:4-25)
    roots = mz_tree.Roots(1, [[0, 1, 2]])
    roots.prepare_no_noise([0.], [[0., 0., 0.]], [-1])
    mm = mz_tree.MinMaxStatsList(1); mm.set_delta(0.01)
    acts = []
    for _ in range(5):
        res = mz_tree.ResultsWrapper(1)
        _, _, la, _ = mz_tree.batch_traverse(roots, 19652, 1.25, 0.997, mm, res, [-1], True)
        acts.append(la[0])
    assert acts == [0] * 5, acts
    print("reference KAT ok", acts)
    import ez_tree
    for name, *args in EZ_CASES:
        case = make_case_ez(ez_tree, *args)
        again = make_case_ez(ez_tree, *args)     # the shimmed reference must be reproducible
        assert all(np.array_equal(case[k], again[k]) for k in case), name
        np.savez_compressed(os.path.join(HERE, f"tree_{name}.npz"), **case)
        print(name, "sum visits ok:", bool((np.where(case["distributions"] < 0, 0, case["distributions"]).sum(1) == case["S"]).all()),
              "resets:", int(case["is_reset"].sum()))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    mz_rand0 = build_ref.load_rand0()
    for name, tree, *args in REUSE_CASES:
        mod = mz_rand0 if tree == "mz" else ez_tree
        case = make_case_reuse(mod, *args)
        again = make_case_reuse(mod, *args)
        assert all(np.array_equal(case[k], again[k]) for k in case), name
        np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **case)
        print(name, "sum visits ok:", bool((np.where(case["distributions"] < 0, 0, case["distributions"]).sum(1) == case["S"]).all()),
              "no-inference marks:", int((case["ix"] == -1).sum()))
    record_random_runs(mz_tree, ez_tree, mz_rand0)


if __name__ == "__main__":
    main()
