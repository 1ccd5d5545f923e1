#!/usr/bin/env python
"""bench.py -- MCTS simulations/s of the fused CUDA search (BASELINE.json metric) on N B200s.

A "step" is one full collect step of the hot path over one batch of synthetic observations:
initial_inference -> root preparation (Dirichlet noise) -> num_simulations x [PUCT traverse ->
recurrent_inference -> expand + backpropagate] -> visit-count / root-value extraction, i.e. what
MuZeroPolicy._forward_collect does between receiving obs and choosing actions
(lzero/policy/muzero.py:749-779).  simulations/s = roots * num_simulations / step time.

  python bench.py [--gpus N --steps K --warmup W]             # our arm  (torchrun for N > 1)
  python bench.py --impl reference [--gpus N --steps K ...]   # reference arm: the reference's own
        CPU path (compiled reference ctree from oracle/_ref + PyTorch-CPU fp32 model) on host cores

One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
_emit = print

METRIC = "MCTS simulations/sec (batched search+infer)"
UNIT = "simulations/s"
# --workload muzero (default): SURVEY.md 8(d) config 3, the north star.  --workload efficientzero: BASELINE.json configs[1]
# (SURVEY 8(f) row f-1) -- 96x96 frames: the reference EfficientZeroModel cannot be constructed for 84x84 with
# downsample=True (efficientzero_model.py:120-126 defines latent_size for 96 and 64 only).
WORKLOADS = {
    "muzero": dict(
        roots=1024, sims=50, actions=18, obs=(4, 84, 84), ez=False,
        name="Atari 84x84 MuZero ResNet (64ch, 1 res block, support 601), num_simulations=50, 1024 roots per GPU, 18 actions",
        # algorithmic FLOPs (SURVEY.md 8d): per root per simulation at P=36, A=18
        flop_recurrent=14_427_392),
    "efficientzero": dict(
        roots=256, sims=50, actions=6, obs=(4, 96, 96), ez=True, lstm_horizon_len=5,
        name="Atari 96x96 EfficientZero ResNet (64ch, 1 res block, LSTM 512, support 601), num_simulations=50, 256 roots per GPU, "
             "6 actions, lstm_horizon_len=5",
        # MuZero count at A=6 (13,928,960) with the reward FC1 (576x32 MAC) replaced by the LSTM step ((576+512) x 2048 MAC)
        # and Linear(512, 32): 2 x (6,964,480 - 18,432 + 2,228,224 + 16,384)
        flop_recurrent=18_381_312),
}
WL = WORKLOADS["muzero"]
ROOTS_PER_GPU = NUM_SIMULATIONS = ACTIONS = OBS = WORKLOAD = FLOP_RECURRENT = None


def select_workload(name):
    global WL, ROOTS_PER_GPU, NUM_SIMULATIONS, ACTIONS, OBS, WORKLOAD, FLOP_RECURRENT
    WL = WORKLOADS[name]
    ROOTS_PER_GPU, NUM_SIMULATIONS, ACTIONS, OBS = WL["roots"], WL["sims"], WL["actions"], WL["obs"]
    WORKLOAD, FLOP_RECURRENT = WL["name"], WL["flop_recurrent"]


select_workload("muzero")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="muzero", choices=sorted(WORKLOADS))
    ap.add_argument("--roots", type=int, default=None)
    ap.add_argument("--sims", type=int, default=None)
    ap.add_argument("--cpu-sample-roots", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong_scaling and extra.workloads blocks")
    ap.add_argument("--h2d-chunks", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's visits, root values, ...) as DIR/<name>.npy; the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    select_workload(args.workload)
    args.roots = args.roots or ROOTS_PER_GPU
    args.sims = args.sims or NUM_SIMULATIONS
    return args


def host_threads():
    """Threads for the reference arm's PyTorch-CPU model: the PHYSICAL cores this process may run on (PyTorch's own default when
    nothing is pinned; one thread per hardware thread of a 2-way SMT host makes the small convolutions of this model collapse --
    measured 17 vs ~5000 simulations/s).  torchrun exports OMP_NUM_THREADS=1 to its workers, which would otherwise starve the
    reference arm at N > 1, so the count is set explicitly."""
    try:
        logical = len(os.sched_getaffinity(0))
    except AttributeError:
        logical = os.cpu_count() or 1
    smt = 1
    try:
        sib = open("/sys/devices/system/cpu/cpu0/topology/thread_siblings_list").read().strip()
        smt = max(1, len([x for part in sib.split(",") for x in ([part] if "-" not in part else range(int(part.split("-")[0]), int(part.split("-")[1]) + 1))]))
    except Exception:
        pass
    return max(1, min(logical // smt, 64))


def make_reference_model(seed=0):
    """Reference arm / cpu_baseline only: the PyTorch-CPU restatement of the reference model (oracle/)."""
    import torch
    from oracle.model_ref import EfficientZeroModelRef, MuZeroModelRef, emulate_trained_
    torch.manual_seed(seed)
    cls = EfficientZeroModelRef if WL["ez"] else MuZeroModelRef
    return emulate_trained_(cls(OBS, ACTIONS), seed)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU pipeline
# ------------------------------------------------------------------------------------------------
def run_reference_pipeline(roots, sims, steps, warmup, threads=None):
    import numpy as np
    import torch
    from oracle.search_ref import SearchRef, SearchRefEZ, collect_step_ref, collect_step_ref_ez, load_tree_module
    threads = threads or host_threads()
    torch.set_num_threads(threads)
    cores = torch.get_num_threads()
    tree, kind = load_tree_module(prefer_ref=True, name="ez_tree" if WL["ez"] else "mz_tree")
    model = make_reference_model()
    # as the reference runs it: stochastic tie-break is irrelevant for timing; keep deterministic.  The
    # duplicated recurrent_inference of mcts_ctree.py:338/:345 is part of the unmodified MuZero driver (the
    # EfficientZero driver, :729-876, calls the network once).
    if WL["ez"]:
        search = SearchRefEZ(tree, lstm_horizon_len=WL["lstm_horizon_len"], num_simulations=sims)
        collect_step_ref = collect_step_ref_ez
    else:
        search = SearchRef(tree, num_simulations=sims, duplicate_inference=True)
    rng = np.random.default_rng(0)
    torch.manual_seed(0)
    times = []
    for it in range(warmup + steps):
        obs = torch.rand(roots, *OBS)
        mask = np.ones((roots, ACTIONS))
        noises = [rng.dirichlet([0.3] * ACTIONS).astype(np.float32).tolist() for _ in range(roots)]
        t0 = time.perf_counter()
        collect_step_ref(search, model, obs, mask, [-1] * roots, noises=noises)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return dict(value=roots * sims / mean, seconds_per_step=mean, cores=cores, nproc=os.cpu_count(), kind="reference" if kind == "reference" else "port",
                sample=f"{roots} roots x {sims} simulations per step ({steps} timed steps after {warmup} warm-up), "
                       f"{'compiled reference ' + ('ez_tree' if WL['ez'] else 'mz_tree') + ' (oracle/_ref)' if kind == 'reference' else 'C port of the ctree'} + "
                       f"PyTorch-CPU fp32 model restatement, "
                       f"{'one recurrent_inference per simulation (mcts_ctree.py:834)' if WL['ez'] else 'duplicate recurrent_inference kept (mcts_ctree.py:338,345)'}, "
                       f"torch threads={cores} (physical cores of this process's affinity mask, capped at 64; the host reports {os.cpu_count()} logical CPUs)")


def reference_arm(args, rank, world):
    if rank != 0:
        return
    roots = args.cpu_sample_roots
    warm = max(3, args.warmup)           # the same warm-up rule as the repo arm
    r = run_reference_pipeline(roots, args.sims, max(1, args.steps), warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": max(1, args.steps), "warmup": warm, "ms_per_step": r["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_roots": roots, "num_simulations": args.sims, "actions": ACTIONS,
                   "note": "the reference's CPU path timed on rank 0's host cores on a bounded sample of the workload (128 of the "
                           "1024 roots per step); the tree is single-threaded by construction, the PyTorch-CPU model uses every core"},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "nproc": r["nproc"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, result):
    """Writes the per-root arrays of one search_batch result as out_dir/<name>.npy in float32 (visit counts are exact there).
    When together they would pass DUMP_LIMIT bytes, the same seeded sample of roots is taken from each and its root
    indices are written as rows.npy."""
    import numpy as np
    arrays = {k: v.cpu().numpy().astype(np.float32) for k, v in result.items()}
    roots = len(arrays["visits"])
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if roots * row_bytes > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(roots, (DUMP_LIMIT - 4096) // (row_bytes + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def _peak():
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
        return float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))), \
            "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
    return 1590.0, "fallback (B200_PROFILING.md: 1.59 PFLOP/s burst)"


def _traffic(workload_key):
    """dram__bytes_read + dram__bytes_write of the dominant kernel from the committed ncu capture (profiles/roofline_traffic.json,
    written by profiles/summarize.py), or None when no capture of the current kernel exists."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        e = t.get(workload_key)
        return (e["bytes_per_launch"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


def ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import lightzero_b200 as lzb
    from lightzero_b200 import cabi
    from lightzero_b200.collect import EfficientZeroCollectPolicy, MuZeroCollectPolicy
    from lightzero_b200.dist import gather_search_results
    from lightzero_b200.synthetic_weights import synthetic_state_dict
    lib = cabi.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        """`warmup` untimed steps, then exactly `steps` steps between barrier + synchronize; CUDA events around every step on
        the launching stream.  Returns (sum of device ms, wall ms, library kernel launches in the timed region)."""
        for i in range(warmup):
            fn(i)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = lib.lz_debug_launch_count()
        t0 = time.perf_counter()
        for i in range(steps):
            ev[i][0].record()
            fn(warmup + i)
            ev[i][1].record()
        barrier()
        wall = time.perf_counter() - t0
        launches = lib.lz_debug_launch_count() - l0
        return sum(a.elapsed_time(b) for a, b in ev), wall * 1e3, launches

    def maxr(*vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def build(wl, B, S):
        """model (synthetic weights in the reference's state_dict layout), collect policy, synthetic inputs for one workload"""
        A, obs_shape, ez = wl["actions"], wl["obs"], wl["ez"]
        sd = synthetic_state_dict(obs_shape, A, efficientzero=ez, seed=0)
        if ez:
            model = lzb.EfficientZeroModel(observation_shape=obs_shape, action_space_size=A, device=dev).load_state_dict(sd)
            policy = EfficientZeroCollectPolicy(model, dict(num_simulations=S, discount_factor=0.997, lstm_horizon_len=wl["lstm_horizon_len"]))
        else:
            model = lzb.MuZeroModel(observation_shape=obs_shape, action_space_size=A, device=dev).load_state_dict(sd)
            policy = MuZeroCollectPolicy(model, dict(num_simulations=S, deterministic=True, discount_factor=0.997))
        policy.h2d_chunks = args.h2d_chunks
        # rotating observation batches so no step re-reads a cached batch; every rank draws its own roots.  Atari frames are
        # uint8 (the emulator's format; the reference scales them to [0, 1] in its env wrapper): the device-resident arm gets
        # them already scaled in HBM as float32, the end-to-end arm uploads the uint8 frames
        g = torch.Generator().manual_seed(1000 + rank)
        NBUF = 3
        h_u8 = [torch.randint(0, 256, (B, *obs_shape), dtype=torch.uint8, generator=g).pin_memory() for _ in range(NBUF)]
        d_f32 = [(h.to(dev).to(torch.float32) / 255.0) for h in h_u8]
        h_mask = torch.ones(B, A, dtype=torch.uint8).pin_memory()
        h_noise = torch.from_numpy(np.random.default_rng(rank).dirichlet([0.3] * A, size=B).astype(np.float32)).pin_memory()
        # end-to-end arm with the collector state on the device (SURVEY 8(f) f-3): the step's host input is ONE new uint8 frame per
        # environment (what the emulator delivers per step, muzero_collector.py:520-545) + the action mask + the root noise
        fs = None
        if not ez and obs_shape[0] == 4:
            from lightzero_b200.collector import FrameStack
            fs = FrameStack(B, obs_shape[0], obs_shape[1], obs_shape[2], device=dev)
            fs.push(h_u8[0][:, 0].contiguous().pin_memory(), reset=torch.ones(B, dtype=torch.uint8).pin_memory())
        h_new = [h[:, -1].contiguous().pin_memory() for h in h_u8]
        return dict(model=model, policy=policy, h_u8=h_u8, d_f32=d_f32, h_mask=h_mask, h_noise=h_noise, fs=fs, h_new=h_new,
                    d_mask=h_mask.to(dev), d_noise=h_noise.to(dev), B=B, S=S, A=A, NBUF=NBUF, wl=wl)

    def device_step(w, gather=True):
        def fn(i):
            r = w["policy"].search_batch(w["d_f32"][i % w["NBUF"]], w["d_mask"], w["d_noise"], None, deterministic=True, read_back=False)
            if world > 1 and gather:   # the only collective of the path: all-gather of the finished results over NCCL
                gather_search_results(r["visits"], r["values"], w["B"] * world)
            w["last"] = r
            return r
        return fn

    def e2e_step(w, full_stack=False):
        if full_stack or w["fs"] is None:      # the whole uint8 observation stack uploaded every step
            return lambda i: w["policy"].search_batch(w["h_u8"][i % w["NBUF"]], w["h_mask"], w["h_noise"], None, deterministic=True, read_back=True)

        def fn(i):                             # frame stacks resident on the device: one new frame per environment per step
            w["fs"].push(w["h_new"][i % w["NBUF"]])
            d_mask = w["h_mask"].to(dev, non_blocking=True)
            d_noise = w["h_noise"].to(dev, non_blocking=True)
            return w["policy"].search_batch(w["fs"].view(), d_mask, d_noise, None, deterministic=True, read_back=True)
        return fn

    def search_only(w):
        """the search() window alone: roots already prepared, latents resident; CUDA events around the graph launch"""
        model, policy, B, S = w["model"], w["policy"], w["B"], w["S"]
        ez = w["wl"]["ez"]
        out0 = model.initial_inference(w["d_f32"][0])
        mcts = policy.mcts
        roots = mcts.roots(B, torch.ones(B, w["A"], dtype=torch.uint8))
        if ez:
            roots._lstm_horizon = w["wl"]["lstm_horizon_len"]
        roots.prepare(0.25, w["d_noise"], None, out0.policy_logits, None)
        mode = (1, w["wl"]["lstm_horizon_len"]) if ez else ()
        roots._materialize(S, mcts._params())
        q = roots._tree.search_for(model, S, mode)
        evs = []
        for i in range(3 + args.steps):
            roots._materialize(S, mcts._params())
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if ez:
                cabi.check(lib.lz_search_run_ez(q, out0.latent_state.data_ptr(), None, None, cabi.stream_ptr()), "lz_search_run_ez")
            else:
                cabi.check(lib.lz_search_run(q, out0.latent_state.data_ptr(), 1, cabi.stream_ptr()), "lz_search_run")
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = sorted(x.elapsed_time(y) for x, y in evs[3:])
        return sum(ms) / len(ms), ms[0], lib.lz_search_num_kernels(q)

    warm = max(3, args.warmup)
    peak_tf, peak_note = _peak()

    # ------------------------------------------------------------------ headline workload (weak scaling: roots per GPU fixed)
    W = build(WL, args.roots, args.sims)
    B, S, A, EZ = W["B"], W["S"], W["A"], WL["ez"]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()      # sampled across warm-up + timed region (same load; nvidia-smi needs ~100 ms to start)
        time.sleep(0.3)
    dev_ms, wall_ms, launches = timed(device_step(W), args.steps, warm)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:     # before the e2e steps reuse the policy's output buffers
        dump_outputs(args.dump_outputs, W["last"])
    e2e_dev_ms, e2e_wall_ms, _ = timed(e2e_step(W), args.steps, warm)
    e2e_full_wall_ms = e2e_wall_ms
    if W["fs"] is not None:
        _, e2e_full_wall_ms, _ = timed(e2e_step(W, full_stack=True), args.steps, warm)
    graph_avg_ms, graph_min_ms, num_kernels_search = search_only(W)
    dev_ms, wall_ms, e2e_dev_ms, e2e_wall_ms, graph_avg_ms, e2e_full_wall_ms = maxr(dev_ms, wall_ms, e2e_dev_ms, e2e_wall_ms, graph_avg_ms, e2e_full_wall_ms)

    # ------------------------------------------------------------------ strong scaling: the north-star split of ONE 1024-root batch
    strong = None
    if not args.no_extras and args.workload == "muzero":
        G = WORKLOADS["muzero"]["roots"]
        if G % world == 0:
            strong = {"global_roots": G, "roots_per_gpu": G // world, "note": "BASELINE configs[2]: the same 1024 roots sharded over the GPUs "
                      "(1024 / N per GPU; no data-path collective, one NCCL all-gather of the results per step); value = 1024 x S / max-over-ranks step time"}
            for S2 in (50, 200):
                if world == 1 and S2 == args.sims and args.roots == G:
                    d_ms, k_ms = dev_ms / args.steps, graph_avg_ms
                else:
                    W2 = build(WORKLOADS["muzero"], G // world, S2)
                    n2 = max(3, min(args.steps, 5))
                    d2, _, _ = timed(device_step(W2), n2, 3)
                    k_ms, _, _ = search_only(W2)
                    d_ms, k_ms = maxr(d2 / n2, k_ms)
                    del W2
                strong[f"S{S2}"] = {"num_simulations": S2, "ms_per_step": d_ms, "value": G * S2 / (d_ms * 1e-3), "unit": UNIT,
                                    "search_only_ms": k_ms}

    # ------------------------------------------------------------------ extra workloads (driver-visible numbers for the other configs)
    extra = None
    if not args.no_extras and args.workload == "muzero":
        wl2 = WORKLOADS["efficientzero"]
        W3 = build(wl2, wl2["roots"], wl2["sims"])
        n3 = max(3, min(args.steps, 5))
        d3, _, _ = timed(device_step(W3), n3, 3)
        e3, ew3, _ = timed(e2e_step(W3), n3, 3)
        k3, _, nk3 = search_only(W3)
        d3, ew3, k3 = maxr(d3 / n3, ew3 / n3, k3)
        tot3 = wl2["roots"] * world
        extra = {"workloads": {"efficientzero": {
            "workload": wl2["name"], "roots_per_gpu": wl2["roots"], "num_simulations": wl2["sims"], "actions": wl2["actions"],
            "ms_per_step": d3, "value": tot3 * wl2["sims"] / (d3 * 1e-3), "unit": UNIT,
            "e2e_value": tot3 * wl2["sims"] / (ew3 * 1e-3), "search_only_ms": k3, "search_graph_kernels": nk3,
            "roofline_frac": wl2["roots"] * wl2["sims"] * wl2["flop_recurrent"] / (k3 * 1e-3) / 1e12 / peak_tf,
            "note": "BASELINE configs[1] (96x96: the reference EfficientZeroModel cannot be built for 84x84 with downsample); roofline_frac = "
                    "algorithmic FLOPs of the search graph / its CUDA-event duration / measured bf16 peak"}}}
        del W3

    if rank == 0:
        total_roots = B * world
        ms_per_step = dev_ms / args.steps
        value = total_roots * S / (ms_per_step * 1e-3)
        e2e_ms = e2e_wall_ms / args.steps          # host-visible time: includes H2D, launch, D2H, final sync
        e2e_value = total_roots * S / (e2e_ms * 1e-3)
        h2d_full = W["h_u8"][0].numel() + W["h_mask"].numel() + W["h_noise"].numel() * 4
        h2d = (W["h_new"][0].numel() + W["h_mask"].numel() + W["h_noise"].numel() * 4) if W["fs"] is not None else h2d_full
        d2h = B * A * 4 + B * 4 * 3 + B * A * 4
        traffic, traffic_src = _traffic(args.workload if (B, S, A) == (WL["roots"], WL["sims"], WL["actions"]) else "none")
        achieved = B * S * FLOP_RECURRENT / (graph_avg_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (fp16x2-split tensor MMAs, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": WORKLOAD, "roots_per_gpu": B, "global_roots": total_roots, "num_simulations": S,
                       "actions": A, "obs": list(OBS), "parallelism": f"roots sharded x{world}, no data-path collective; one NCCL all-gather of visits/values per step",
                       "step": "initial_inference + prepare + S x (traverse, recurrent_inference, backpropagate) + results"
                               + (" (EfficientZero: value-prefix trees, LSTM state reset every lstm_horizon_len steps)" if EZ else ""),
                       "deterministic": True,
                       "math": "tcgen05 fp16 hi/lo split (fp32-accurate: A_hi x [B_hi | B_lo] as one N = 128 MMA + A_lo x B_hi, fp32 accumulate in TMEM): the 1e-5 parity mode",
                       "weights": "random, reference state_dict layout (lightzero_b200.synthetic_weights; no checkpoints offline)",
                       "l2": f"no explicit flush: per-step working set = rotating 3 x {W['d_f32'][0].numel() * 4 / 1e6:.0f} MB observation batches + "
                             f"{(S + 1) * B * (2304 + (1024 if EZ else 0)) * 4 / 1e6:.0f} MB latent / LSTM-state pools > 126 MB L2",
                       "search_only_ms": graph_avg_ms,
                       "search_only_sims_per_s": total_roots * S / (graph_avg_ms * 1e-3),
                       "wall_ms_per_step": wall_ms / args.steps},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "device_ms_per_step": e2e_dev_ms / args.steps,
                    "api": (f"lightzero_b200.collector.FrameStack.push (ONE new pinned host uint8 frame per environment per step, the emulator's "
                            f"per-step output; the {OBS[0]}-frame stacks of GameSegment.get_obs stay on the device) + mask / noise uploads + "
                            f"lightzero_b200.collect.{type(W['policy']).__name__}.search_batch (lz_search_collect_u8; pinned host visits / values out); "
                            "the frames are scaled to [0, 1] inside the first conv kernel exactly like the reference's ScaledFloatFrameWrapper")
                           if W["fs"] is not None else
                           (f"lightzero_b200.collect.{type(W['policy']).__name__}.search_batch (pinned host uint8 frames / mask / noise in, pinned host "
                            f"visits / values out; lz_search_collect_host_u8, {args.h2d_chunks} overlapped H2D chunks)"),
                    "full_stack_upload": {"value": total_roots * S / (e2e_full_wall_ms / args.steps * 1e-3), "ms_per_step": e2e_full_wall_ms / args.steps,
                                          "h2d_bytes_per_step": h2d_full,
                                          "note": f"the same step with the whole {OBS[0]}-frame uint8 stack uploaded every step (lz_search_collect_host_u8, "
                                                  f"{args.h2d_chunks} overlapped H2D chunks): what a collector without device-resident frame stacks pays"}},
            "gpu_launches": int(launches),
            "gpu_launches_note": "counted by the library (lz_debug_launch_count: every kernel it enqueues, graph kernel nodes included) over the timed region",
            "search_graph_kernels": num_kernels_search,
            "roofline": {"bound": "tensor",
                         "kernel": ("search graph = 1 + num_simulations x [k_net_tc conv trunk + prediction heads (tcgen05), k_ez_lstm_tc (tcgen05 3xFP16 GEMM "
                                    "over all roots + cell update), k_ez_head, tree back-up + descent]" if EZ else
                                    "k_net_tc, persistent launch = num_simulations x [tree back-up/descent + fused recurrent_inference] (tcgen05)"),
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "frac_of_peak_over_3": 3 * achieved / peak_tf,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_note, "kernel_ms": graph_avg_ms, "kernel_ms_min": graph_min_ms,
                         "kernel_share_of_step": graph_avg_ms / ms_per_step,
                         "flop_per_launch": B * S * FLOP_RECURRENT,
                         "issued_flop_per_launch": int(B * S * FLOP_RECURRENT * 3 * 384 / 252) if not EZ else None,
                         "note": ("achieved = algorithmic FLOPs (18,381,312 per root per simulation: the MuZero count at A=6 with the reward FC1 replaced "
                                  "by the LSTM step and Linear(512,32)) x roots x simulations / CUDA-event duration of the whole search graph, against the "
                                  "measured bf16 peak") if EZ else "achieved = algorithmic FLOPs (SURVEY 8d, 14,427,392 per root per simulation, counted ONCE) x roots x "
                                 "simulations / CUDA-event duration of the persistent launch (which also contains the tree phases), against "
                                 "the measured bf16 peak.  The kernel issues 3 fp16 products per MAC (fp32-accurate hi/lo split) on 384 padded "
                                 "rows per 252 real ones = 4.57x the algorithmic FLOPs: the ceiling of this formulation is 21.9% of the tensor peak; "
                                 "frac_of_peak_over_3 is SURVEY 8d's alternative bookkeeping (1x algorithmic FLOPs against peak / 3)"},
        }
        if strong:
            line["strong_scaling"] = strong
        if extra:
            line["extra"] = extra
        if not args.no_cpu_baseline and world == 1:
            r = run_reference_pipeline(args.cpu_sample_roots, S, 1, 0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "nproc": r["nproc"], "kind": r["kind"], "sample": r["sample"]}
        _emit(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # stdout must carry exactly ONE JSON line: libraries (e.g. NCCL's version banner) write to fd 1, so park the
    # real stdout and point fd 1 at stderr until the result is printed
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit

    def _emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (line + "\n").encode())
    args = parse()
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1 to its workers: give the reference arm every core this process may run on
        n = str(host_threads())
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ[k] = n
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
