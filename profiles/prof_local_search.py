"""Whole-episode replay and local search (profiles/README.md, "Whole-episode replay and local search").

  (a) mtfjsp_replay of complete random-rollout sequences (T = N, one candidate per env, src = arange) at 65,536 J6M6E2,
      16,384 J10M10E3 and 4,096 J30M20E5 envs (left shift on), through the C entry point into preallocated outputs: CUDA
      events around each call, L2 overwritten (256 MB memset) before every timed call, median of 10 calls after 2
      untimed ones.  Against the composition producing the same costs: mtfjsp_gather of every env from a freshly reset
      handle, N x mtfjsp_step, mtfjsp_costs; events around the whole composition, L2 overwritten before it, median of 3
      after 1 untimed one.  Both outputs (costs, summed rewards, first invalid index) are compared in the same run.
      Rate: env-steps/s = envs x N / time.
  (b) local_search (full neighbourhood, steepest descent to a local optimum or 200 rounds) on the 100 shipped J6M6E2
      test instances from greedy `iotj` / `n12800` (tf32), GREEDY_R (no left shift, as the rule rows run) and beam
      W = 32 with both checkpoints: mean objective and mean weighted gap to the MIP row (csv13) before and after, rounds
      run, wall time of the search (host clock, ends in a synchronise).  Plus one max_neighbours-sampled run at J30M20E5
      on 128 device-generated instances (1,024 sampled neighbours each, 5 rounds) from random-rollout sequences.
Prints the results as JSON and writes them to the path given as the first argument (default
profiles/local_search_b200.json)."""
import ctypes as C
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
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
GOLD = os.path.join(ROOT, "tests", "golden")
SIZES = [(65536, 6, 6, 2), (16384, 10, 10, 3), (4096, 30, 20, 5)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi name,power.limit,clocks.sm,clocks.max.sm": q.stdout.strip()}


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def ev_time(fn, flush):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3


def ptr(x):
    return C.c_void_p(x.data_ptr())


def fresh_env(d, w, B, J, M, E):
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    env.obs()
    return env


def replay_vs_composition(B, J, M, E, flush):
    lib = envm._lib.lib()
    N = J * M
    d = ins.device_instances(0, B, J, M, E, seed=91)
    w = ins.random_weights(0, B, 91)
    env = fresh_env(d, w, B, J, M, E)
    acts = []
    for _ in range(N):
        env.random_step(seed=13)
        acts.append(torch.stack((env.op, env.mach), 1).clone())
    acts = torch.stack(acts)                                                   # [N,B,2]
    fresh = fresh_env(d, w, B, J, M, E)
    cp = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    dev = env.device
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    src = torch.arange(B, dtype=torch.int32, device=dev)
    act_rt = acts.transpose(0, 1).contiguous()                                 # [B,N,2]
    f4 = torch.empty((B, 4), dtype=torch.float64, device=dev)
    r5 = torch.empty((B, 5), dtype=torch.float64, device=dev)
    fi = torch.empty((B,), dtype=torch.int32, device=dev)
    call = lambda: envm.check(lib.mtfjsp_replay(env._h, ptr(src), B, ptr(act_rt), N, ptr(f4), ptr(r5), ptr(fi), s),
                              "mtfjsp_replay")
    for _ in range(2):
        call()
    t_rep = [ev_time(call, flush) for _ in range(10)]
    ops = [acts[k, :, 0].contiguous() for k in range(N)]
    machs = [acts[k, :, 1].contiguous() for k in range(N)]
    c4 = torch.empty((B, 4), dtype=torch.float64, device=dev)
    c5 = torch.empty((B, 5), dtype=torch.float64, device=dev)
    cinv = torch.empty((B,), dtype=torch.uint8, device=dev)

    def compose(tot=None, first=None):
        envm.check(lib.mtfjsp_gather(cp._h, fresh._h, ptr(src), s), "mtfjsp_gather")
        for k in range(N):
            envm.check(lib.mtfjsp_step(cp._h, ptr(ops[k]), ptr(machs[k]), ptr(c5), None, None, ptr(cinv), s), "mtfjsp_step")
            if tot is not None:
                tot += c5
                first.copy_(torch.where((first < 0) & (cinv != 0), k, first))
        envm.check(lib.mtfjsp_costs(cp._h, ptr(c4), None, s), "mtfjsp_costs")

    tot = torch.zeros((B, 5), dtype=torch.float64, device=dev)
    first = torch.full((B,), -1, dtype=torch.int32, device=dev)
    compose(tot, first)
    same = bool(torch.equal(f4, c4) and torch.equal(r5, tot) and torch.equal(fi, first))
    t_cmp = [ev_time(compose, flush) for _ in range(3)]
    tr, tc = float(np.median(t_rep)), float(np.median(t_cmp))
    out = {"envs": B, "J": J, "M": M, "E": E, "T": N, "env_steps": B * N,
           "replay_s": tr, "replay_s_runs": t_rep, "replay_env_steps_per_s": B * N / tr,
           "composition_s": tc, "composition_s_runs": t_cmp, "composition_env_steps_per_s": B * N / tc,
           "speedup": tc / tr, "outputs_equal": same, "all_valid": bool((fi == -1).all().item())}
    for e in (env, fresh, cp):
        e.close()
    return out


def mip_dict(c):
    return {"Makespan": c[:, 0], "MachineEC": c[:, 1], "TransEC": c[:, 2], "MachineIdleT": c[:, 3]}


def searched(name, inst, actions, start_final4, mip, left_shift):
    t, out = wall(lambda: search.local_search(inst, actions, left_shift=left_shift, rounds=200))
    start_obj = val._objective(start_final4, (0.4, 0.4, 0.2))
    assert np.array_equal(out["history"][0], start_obj), name
    row = {"start": name, "left_shift": left_shift, "mean_objective_before": float(start_obj.mean()),
           "mean_objective_after": float(out["objective"].mean()),
           "mean_mip_gap_before": float(val.mip_gaps(start_final4, mip)[1].mean()),
           "mean_mip_gap_after": float(val.mip_gaps(out["final4"], mip)[1].mean()),
           "instances_improved": int((out["objective"] < start_obj).sum()),
           "rounds_run": int(out["accepted"].shape[0]), "wall_s": t}
    print(json.dumps(row), flush=True)
    return row


def quality():
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    mip = mip_dict(np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv13"])
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    rows = []
    for tag in ("iotj", "n12800"):
        sd_op, sd_m = val.load_actor_state_dicts(g, tag)
        ja, ma = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")
        gr = val.greedy_validate(ja, ma, inst, return_actions=True)
        rows.append(searched("greedy %s tf32" % tag, inst, gr["actions"], gr["final4"], mip, True))
        bm = val.beam_validate(ja, ma, inst, 32, return_actions=True)
        rows.append(searched("beam W=32 %s tf32" % tag, inst, bm["best_actions"], bm["best_final4"], mip, True))
    env = envm.BatchedMTFJSPEnv(100, 6, 6, 2, left_shift=False, obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (100, 1)))
    acts = rules.greedy_reward_rollout(env)
    rows.append(searched("GREEDY_R", inst, acts.cpu().numpy(), env.costs().cpu().numpy(), mip, False))
    env.close()
    return rows


def sampled_j30m20(S=128, K=1024, rounds=5):
    J, M, E = 30, 20, 5
    d = ins.device_instances(0, S, J, M, E, seed=404)
    inst = {k: v.cpu().numpy() for k, v in d.items()}
    env = fresh_env(d, np.tile([0.4, 0.4, 0.2], (S, 1)), S, J, M, E)
    acts = []
    for _ in range(J * M):
        env.random_step(seed=17)
        acts.append(torch.stack((env.op, env.mach), 1).clone())
    start = val._objective(env.costs().cpu().numpy(), (0.4, 0.4, 0.2))
    env.close()
    t, out = wall(lambda: search.local_search(inst, torch.stack(acts), rounds=rounds, max_neighbours=K, seed=1))
    row = {"instances": "device J30M20E5", "S": S, "start": "random rollout", "max_neighbours": K,
           "rounds": int(out["accepted"].shape[0]), "mean_objective_before": float(start.mean()),
           "mean_objective_after": float(out["objective"].mean()), "wall_s": t,
           "replays": int(out["accepted"].shape[0]) * S * K}
    print(json.dumps(row), flush=True)
    return row


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "local_search_b200.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res["replay"] = []
    for B, J, M, E in SIZES:
        res["replay"].append(replay_vs_composition(B, J, M, E, flush))
        print(json.dumps(res["replay"][-1]), flush=True)
    del flush
    torch.cuda.empty_cache()
    res["local_search_shipped_100"] = quality()
    res["local_search_sampled"] = sampled_j30m20()
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(txt)


if __name__ == "__main__":
    main()
