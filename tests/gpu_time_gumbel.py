"""Times the Gumbel MuZero search against the MuZero searches that use the same network kernels, in one process with CUDA
events after warm-up (B = 1024 roots, S = 50 simulations, A = 18, tcgen05 tc3 conv model at 84x84, synthetic weights):
  * Gumbel fused search (lz_search_run_gumbel) with m = 4 and m = 18;
  * MuZero multi-launch search ([traverse] + S x [network, back-up + traverse], the same graph shape);
  * MuZero persistent search (one tcgen05 launch, tree_persist.cuh);
plus the tree kernels' time per simulation (torch.profiler kernel records) and the reference Gumbel CPU pipeline (compiled
gmz_tree + PyTorch CPU model) on a 128-root sample.  Prints one JSON line (card name and power limit included).

    python tests/gpu_time_gumbel.py > profiles/gumbel_time.json
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lightzero_b200 as lzb  # noqa: E402
from lightzero_b200.synthetic_weights import synthetic_state_dict  # noqa: E402

B, S, A = 1024, 50, 18
REPS = int(os.environ.get("GMZ_REPS", 10))


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in line.split(",")]
        return name, power
    except Exception as e:       # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    name, power = gpu_info()
    sd = synthetic_state_dict((4, 84, 84), A)
    model = lzb.MuZeroModel(observation_shape=(4, 84, 84), action_space_size=A).load_state_dict(sd)
    model.set_math(1)
    dev = torch.device("cuda", torch.cuda.current_device())
    obs = torch.rand(B, 4, 84, 84, device=dev)
    out = model.initial_inference(obs)
    rng = np.random.default_rng(0)
    noise = torch.from_numpy(rng.dirichlet([0.3] * A, size=B).astype(np.float32)).to(dev)
    values = torch.from_numpy(rng.standard_normal(B).astype(np.float32)).to(dev)
    mask = torch.ones(B, A, dtype=torch.uint8)

    gm = {m: lzb.GumbelMuZeroMCTSCtree(dict(num_simulations=S, max_num_considered_actions=m, discount_factor=0.997)) for m in (4, 18)}
    mz = lzb.MuZeroMCTSCtree(dict(num_simulations=S, deterministic=True, discount_factor=0.997))
    # every variant keeps its own Roots (hence its own device tree and captured graph) alive for the whole run
    roots = {("gumbel", m): gm[m].roots(B, mask) for m in (4, 18)}
    roots["muzero_multi"] = mz.roots(B, mask)
    roots["muzero_persistent"] = mz.roots(B, mask)

    def run(key):
        r = roots[key]
        if key[0] == "gumbel":
            r.prepare(0.25, noise, None, values, out.policy_logits, None)
            gm[key[1]].search(r, model, out.latent_state, None)
        else:
            r.prepare(0.25, noise, None, out.policy_logits, None)
            mz.search(r, model, out.latent_state, None)

    os.environ["LZ_NO_PERSIST"] = "1"          # read when the graph is captured (first run of that search)
    run("muzero_multi")
    del os.environ["LZ_NO_PERSIST"]
    run("muzero_persistent")
    keys = [("gumbel", 4), ("gumbel", 18), "muzero_multi", "muzero_persistent"]
    for k in keys:
        run(k)
    torch.cuda.synchronize()
    ms = {k: [] for k in keys}
    for _ in range(REPS):
        for k in keys:                           # alternating, so drift hits every variant alike
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run(k)
            b.record()
            torch.cuda.synchronize()
            ms[k].append(a.elapsed_time(b))

    def label(k):
        return f"gumbel_m{k[1]}" if isinstance(k, tuple) else k
    res = dict(gpu=name, power_limit=power, B=B, S=S, A=A, model="MuZeroModel 84x84 tc3 (synthetic weights)", reps=REPS,
               search_ms_median={label(k): float(np.median(v)) for k, v in ms.items()},
               search_ms_min={label(k): float(np.min(v)) for k, v in ms.items()})

    # tree kernels per simulation: profiler kernel records of 3 searches per variant
    from torch.profiler import ProfilerActivity, profile
    per_sim = {}
    for k in keys[:3]:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                run(k)
            torch.cuda.synchronize()
        tree_us = net_us = 0.0
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            dur = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            if "k_gmz_" in e.name or "k_tree_" in e.name:
                tree_us += dur
            elif e.name.startswith("k_") or "tc" in e.name:
                net_us += dur
        per_sim[label(k)] = dict(tree_us_per_sim=tree_us / (3 * S), other_kernels_us_per_sim=net_us / (3 * S))
    res["kernel_us_per_simulation"] = per_sim

    # reference Gumbel CPU pipeline (compiled gmz_tree + PyTorch CPU fp32 model), 128 roots
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import make_gumbel_golden as mg
        from oracle.model_ref import MuZeroModelRef
        from oracle.gumbel_ref import GumbelSearchRef, gumbel_search_step_ref
        gmz = mg.load_reference()
        if gmz is not None:
            n = 128
            ref = MuZeroModelRef((4, 84, 84), A)
            ref.load_state_dict({k: v.cpu() for k, v in sd.items()}, strict=False)
            legal = [list(range(A))] * n
            noises = [rng.dirichlet([0.3] * A).astype(np.float32).tolist() for _ in range(n)]
            t0 = time.perf_counter()
            gumbel_search_step_ref(GumbelSearchRef(gmz, num_simulations=S, max_num_considered_actions=4), ref,
                                   obs[:n].cpu(), legal, noises, [-1] * n)
            sec = time.perf_counter() - t0
            res["reference_cpu_128_roots"] = dict(seconds=sec, ms_per_root=1e3 * sec / n, threads=torch.get_num_threads())
    except Exception as e:       # noqa: BLE001
        res["reference_cpu_128_roots"] = f"not run: {e!r}"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
