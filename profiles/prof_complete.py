"""Episode completion on the device and the pilot method on it (profiles/README.md, "Episode completion").

  (a) Completion throughput: mtfjsp_complete with the random base, one candidate per env, left shift on, ESA mask, at
      65,536 J6M6E2, 16,384 J10M10E3 and 4,096 J30M20E5 device-generated envs, from the reset state and from
      mid-episode (after N/2 random steps).  Against the composition it restates (gather into a B-env handle, then
      policy_random + step until done) and against replay of the same whole sequences from the episode start.  CUDA
      events, median of 5 after 1 untimed call; env-steps are the steps the completion takes.  The three final costs are
      compared in the same run.
  (b) pilot_search on the 100 shipped J6M6E2 test instances (tests/golden/pdr_golden.npz), weights 0.4/0.4/0.2, no left
      shift, FINISHED mask: every static rule pair as the base with candidates "all" and "rule", and the random base with
      samples 1 and 8.  Mean objective against the rule's row, GREEDY_R (evaluate_rules) and greedy `iotj` (tf32 actors
      of policy_golden.npz, greedy_validate's defaults), all computed here; wall time (host clock around a call that ends
      in a synchronise), completions and env-steps.
Prints the results as JSON and writes them to the path given as the first argument (default profiles/complete_b200.json)."""
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
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
GOLD = os.path.join(ROOT, "tests", "golden")
W = (0.4, 0.4, 0.2)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi name,power.limit,clocks.sm,clocks.max.sm": q.stdout.strip()}


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


def make_env(B, J, M, E, seed):
    d = ins.synthetic_instances(0, B, J, M, E, seed=seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed=seed))
    return env


def throughput(B, J, M, E):
    N = J * M
    env = make_env(B, J, M, E, 7)
    cp = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    src = torch.arange(B, dtype=torch.int32, device=env.device)
    out = []
    prefix = []
    for start in ("reset", "mid-episode"):
        if start == "mid-episode":
            for _ in range(N // 2):
                env.random_step(seed=3)
                prefix.append(torch.stack((env.op, env.mach), 1).clone())
        k = len(prefix)
        f4, _, fi, ba = env.complete(src, base="random", seed=11)

        def composition():
            cp.gather_from(env, src)
            for _ in range(N - k):
                cp.policy_random(11, 0)
                cp.step(cp.op, cp.mach)

        seqs = torch.cat((torch.stack(prefix), ba[:N - k])) if prefix else ba  # the whole sequences from the start
        t_c = ev_median(lambda: env.complete(src, base="random", seed=11))
        t_g = ev_median(composition)
        t_r = ev_median(lambda: env.replay(seqs))
        composition()
        eq_comp = bool((cp.costs() == f4).all())
        eq_rep = bool((env.replay(seqs)[0] == f4).all())
        steps = B * (N - k)
        out.append({"size": "J%dM%dE%d" % (J, M, E), "envs": B, "start": start, "steps_per_env": N - k,
                    "complete_s": t_c, "composition_s": t_g, "replay_s": t_r,
                    "complete_env_steps_per_s": steps / t_c, "composition_env_steps_per_s": steps / t_g,
                    "replay_env_steps_per_s": B * N / t_r,
                    "composition_over_complete": t_g / t_c, "replay_over_complete": t_r / t_c,
                    "final4_equal_composition": eq_comp, "final4_equal_replay": eq_rep,
                    "all_valid": bool((fi == -1).all())})
        print(json.dumps(out[-1]), flush=True)
    env.close()
    cp.close()
    return out


def pilot_table():
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k] for k in ("t", "p", "transT", "edge")}
    S = 100
    names = [str(x) for x in g["rule_names"]]
    rule_obj = {n: float(val._objective(g["gold"][r], W).mean()) for r, n in enumerate(names)}
    gr = rules.evaluate_rules(g["t"], g["p"], g["transT"], g["edge"], 6, 6, 2, op_rules=(), joint_rules=("GREEDY_R",))
    greedy_r = float(gr["objective"][0].mean())
    op_sd, mch_sd = val.load_actor_state_dicts(os.path.join(GOLD, "policy_golden.npz"), "iotj")
    ja, ma = enc.JobActor(op_sd, 6, 6, precision="tf32"), enc.MachineActor(mch_sd, 6, precision="tf32")
    iotj = float(val._objective(val.greedy_validate(ja, ma, inst, return_actions=True)["final4"], W).mean())
    search.pilot_search({k: v[:2] for k, v in inst.items()}, base=("FIFO", "SPT"))          # module load, warm-up
    rows = []
    runs = [(tuple(n.split("+")), c, 1) for n in names for c in ("all", "rule")] + [("random", "all", q) for q in (1, 8)]
    for base, cand, q in runs:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = search.pilot_search(inst, base=base, candidates=cand, samples=q, seed=0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        name = "+".join(base) if isinstance(base, tuple) else "random"
        h = out["history"]
        row = {"base": name, "candidates": cand, "samples": q, "mean_objective": float(out["objective"].mean()),
               "mean_base_objective": float(out["base_objective"].mean()),
               "rule_row_mean": rule_obj.get(name), "wall_s": dt, "completions": out["completions"],
               "env_steps": out["env_steps"], "history_non_increasing": bool((np.diff(h, axis=0) <= 0).all()),
               "instances_better_than_base": int((out["objective"] < out["base_objective"]).sum()),
               "instances_better_than_greedy_r": int((out["objective"] < gr["objective"][0]).sum())}
        rows.append(row)
        print(json.dumps(row), flush=True)
    return {"instances": S, "greedy_r_mean": greedy_r, "iotj_greedy_mean": iotj, "rule_rows": rule_obj, "runs": rows}


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "complete_b200.json")
    res = {"gpu": gpu_info()}
    res["a_throughput"] = []
    for B, J, M, E in ((65536, 6, 6, 2), (16384, 10, 10, 3), (4096, 30, 20, 5)):
        res["a_throughput"] += throughput(B, J, M, E)
        torch.cuda.empty_cache()
    res["b_pilot"] = pilot_table()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
