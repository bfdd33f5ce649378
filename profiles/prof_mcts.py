"""Monte Carlo tree search on the episode completion (profiles/README.md, "MCTS on the completion").

  (a) On the 100 shipped J6M6E2 test instances (tests/golden/pdr_golden.npz), weights 0.4/0.4/0.2, no left shift,
      FINISHED mask, candidates "all": mcts_search with the MWKR_T+SPT, FIFO+SPT and random bases for c in {0.25, 1, 4}
      at the pilot method's completion count (36 selections a decision, one round of 36 leaves) and at four times that
      (144: four rounds of 36), against pilot_search at the same counts (the priority pilots at 1x only; the random pilot
      with samples 1 and 4).  Mean objective, completions and wall time (host clock around a call that ends in a
      synchronise).
  (b) Device time by kernel in one mcts_search run of 1,024 J10M10E3 generated instances (64 selections, one round a
      decision), from torch.profiler: mtfjsp_mcts_select / mtfjsp_mcts_backup against complete_kernel.  Then the cost of
      padding: one complete call of 65,536 mid-episode J10M10 rows whose paths have depths 0..8 padded to 8, against
      the same rows completed in one call per depth at their own depths (CUDA events, median of 5).
  (c) mcts_search at scale on device-generated instances: 1,024 J10M10E3 at the default budget (256 selections, leaves
      64) and 256 J30M20E5 at 16 selections (one round of 16), default max_nodes: wall time, pool nodes used and the pool's
      memory (36 bytes a node).
Prints the results as JSON and writes them to the path given as the first argument (default profiles/mcts_b200.json)."""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
GOLD = os.path.join(ROOT, "tests", "golden")
NODE_BYTES = 7 * 4 + 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi name,power.limit,clocks.sm,clocks.max.sm": q.stdout.strip()}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def ev_median(fn, runs=5, warm=1):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts))


def table():
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k] for k in ("t", "p", "transT", "edge")}
    search.mcts_search({k: v[:2] for k, v in inst.items()}, simulations=8, leaves=8)        # module load, warm-up
    search.pilot_search({k: v[:2] for k, v in inst.items()})
    rows = []
    for base in (("MWKR_T", "SPT"), ("FIFO", "SPT"), "random"):
        name = "+".join(base) if isinstance(base, tuple) else "random"
        for mult in (1, 4):
            if isinstance(base, tuple) and mult > 1:
                pilot = None
            else:
                pilot, dt = timed(lambda: search.pilot_search(inst, base=base, samples=mult) if base == "random"
                                  else search.pilot_search(inst, base=base))
                rows.append({"method": "pilot", "base": name, "budget": mult, "mean_objective": float(pilot["objective"].mean()),
                             "mean_base_objective": float(pilot["base_objective"].mean()), "completions": pilot["completions"],
                             "wall_s": dt})
                print(json.dumps(rows[-1]), flush=True)
            for c in (0.25, 1.0, 4.0):
                out, dt = timed(lambda: search.mcts_search(inst, base=base, simulations=36 * mult, leaves=36, c=c))
                row = {"method": "mcts", "base": name, "budget": mult, "c": c, "mean_objective": float(out["objective"].mean()),
                       "mean_base_objective": float(out["base_objective"].mean()), "completions": out["completions"],
                       "env_steps": out["env_steps"], "wall_s": dt, "max_nodes_used": int(out["nodes"].max()),
                       "history_non_increasing": bool((np.diff(out["history"], axis=0) <= 0).all())}
                if pilot is not None:
                    row["instances_better_than_pilot"] = int((out["objective"] < pilot["objective"]).sum())
                    row["instances_worse_than_pilot"] = int((out["objective"] > pilot["objective"]).sum())
                rows.append(row)
                print(json.dumps(row), flush=True)
    return rows


def generated(S, J, M, E, seed=7):
    d = ins.synthetic_instances(0, S, J, M, E, seed=seed)
    return {k: d[k] for k in ("t", "p", "transT", "edge")}


def kernel_shares():
    inst = generated(1024, 10, 10, 3)
    search.mcts_search({k: v[:4] for k, v in inst.items()}, simulations=64, leaves=64)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        search.mcts_search(inst, simulations=64, leaves=64)
        torch.cuda.synchronize()
    by = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA":
            by[e.key] = by.get(e.key, 0.0) + e.device_time_total * 1e-6
    total = sum(by.values())
    groups = {"select": sum(v for k, v in by.items() if "mcts_select" in k),
              "backup": sum(v for k, v in by.items() if "mcts_backup" in k),
              "complete": sum(v for k, v in by.items() if "complete_kernel" in k)}
    groups["other"] = total - sum(groups.values())
    return {"instances": "1024 x J10M10E3", "simulations": 64, "leaves": 64, "device_s": groups,
            "share": {k: v / total for k, v in groups.items()},
            "top": sorted(([k, v] for k, v in by.items()), key=lambda x: -x[1])[:8]}


def padding_cost():
    B, J, M, E = 1024, 10, 10, 3
    N = J * M
    d = ins.synthetic_instances(0, B, J, M, E, seed=3)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=False, obs_dtype=torch.float32, mask_mode=envm.MASK_FINISHED)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed=3))
    for _ in range(N // 2):
        env.random_step(seed=9, mask_mode=envm.MASK_FINISHED)
    R, T = 64 * B, 8
    src = (torch.arange(R, device=env.device) // 64).to(torch.int32)
    _, _, _, seqs = env.complete(src, base="random", seed=5, mask_mode=envm.MASK_FINISHED)
    depth = torch.as_tensor(np.random.default_rng(1).integers(0, T + 1, R), device=env.device)
    steps = torch.arange(T, device=env.device)[:, None, None]
    padded = torch.where(steps < depth[None, :, None], seqs[:T], -1)
    groups = [(dd, (depth == dd).nonzero(as_tuple=True)[0]) for dd in range(T + 1)]
    parts = [(src[i].contiguous(), seqs[:dd, i].contiguous() if dd else None) for dd, i in groups]

    def one():
        env.complete(src, padded, base="random", seed=7, mask_mode=envm.MASK_FINISHED)

    def per_depth():
        for s_, a_ in parts:
            env.complete(s_, a_, base="random", seed=7, mask_mode=envm.MASK_FINISHED)

    t_pad, t_own = ev_median(one), ev_median(per_depth)
    env.close()
    return {"rows": R, "size": "J10M10E3 mid-episode (50 ops left)", "depths": "uniform 0..8", "padded_s": t_pad,
            "own_depth_calls_s": t_own, "padded_over_own": t_pad / t_own,
            "mean_pad_steps_per_row": float((T - depth).float().mean())}


def scale():
    out = []
    for S, J, M, E, sims, leaves in ((1024, 10, 10, 3, 256, 64), (256, 30, 20, 5, 16, 16)):
        inst = generated(S, J, M, E)
        search.mcts_search({k: v[:2] for k, v in inst.items()}, simulations=leaves, leaves=leaves)
        res, dt = timed(lambda: search.mcts_search(inst, simulations=sims, leaves=leaves))
        row = {"instances": "%d x J%dM%dE%d" % (S, J, M, E), "simulations": sims, "leaves": leaves,
               "max_nodes": 65536, "wall_s": dt, "completions": res["completions"], "env_steps": res["env_steps"],
               "nodes_used_max": int(res["nodes"].max()), "nodes_used_mean": float(res["nodes"].mean()),
               "pool_bytes": S * 65536 * NODE_BYTES, "mean_objective": float(res["objective"].mean()),
               "mean_base_objective": float(res["base_objective"].mean())}
        out.append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "mcts_b200.json")
    res = {"gpu": gpu_info()}
    res["a_table"] = table()
    res["b_kernel_shares"] = kernel_shares()
    print(json.dumps(res["b_kernel_shares"]), flush=True)
    res["b_padding"] = padding_cost()
    print(json.dumps(res["b_padding"]), flush=True)
    res["c_scale"] = scale()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
