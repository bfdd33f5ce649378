"""Tabu search on the neighbour replay (profiles/README.md, "Tabu search on the neighbour replay").

  (d) Tenure sweep, run first: tabu_search (500 iterations, full neighbourhood, left shift on) on 64 device-generated
      J6M6E2 instances (instances.device_instances, seed 515) from random-rollout sequences, for tenure_mach in
      {0, 5, 20} x tenure_ins in {0, 5, 10, 20, 35, 50, 80}: mean best objective.  (b) and (c) run search's defaults
      (search.TENURE_MACH, search.TENURE_INS), which this sweep chose.
  (a) mtfjsp_replay_moves against the materialised path (search.apply_moves, then mtfjsp_replay) on the same moves of
      random-rollout base sequences: the full neighbourhoods of 100 J6M6E2 and 32 J10M10E3 device-generated instances,
      and 1,024 sampled neighbours of each of 16 J30M20E5 instances, at most 65,536 candidates (one call).  CUDA events,
      L2 overwritten (256 MB memset) before every timed call, median of 10 after 2 untimed ones; the materialised time
      includes apply_moves.  Bytes: the neighbour sequences the materialised path writes and reads again (2 x R x N x 8)
      against the move list replay_moves reads (R x 16).  Output hashes of both paths are compared in the same run.
  (b) On the 100 shipped J6M6E2 test instances, tabu_search at 200 and 1,000 iterations from greedy `iotj` /
      `n12800` (tf32), beam W = 32 of both and GREEDY_R (no left shift, as the rule rows run), against local_search (to
      its optimum, at most 200 rounds) from the same starts: mean objective, mean validate.mip_gaps gap to the MIP row
      (csv13), instances strictly better than local_search, wall time (host clock ending in a synchronise), replays.
  (c) One iteration's device time split into neighbour_moves (torch), replay_moves and the decision (objective, segment
      offsets, mtfjsp_tabu_move): CUDA events around each part, medians over iterations 100 .. 199 of a run from
      greedy `iotj` on the shipped instances; with the share of reassignments among the moves taken and the number of
      distinct current objectives an instance visits over those 100 iterations.
Prints the results as JSON and writes them to the path given as the first argument (default profiles/tabu_b200.json)."""
import hashlib
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
W = (0.4, 0.4, 0.2)
TENURES_MACH = (0, 5, 20)
TENURES_INS = (0, 5, 10, 20, 35, 50, 80)


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


def fresh_env(d, S, J, M, E, left_shift=True):
    env = envm.BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(W), (S, 1)))
    env.obs()
    return env


def random_starts(S, J, M, E, seed):
    """Device-generated instances (as numpy) and one random-rollout sequence each ([N,S,2] on the device)."""
    d = ins.device_instances(0, S, J, M, E, seed=seed)
    env = fresh_env(d, S, J, M, E)
    acts = []
    for _ in range(J * M):
        env.random_step(seed=seed)
        acts.append(torch.stack((env.op, env.mach), 1).clone())
    env.close()
    return {k: v.cpu().numpy() for k, v in d.items()}, torch.stack(acts)


def tenure_sweep(S=64, iterations=500):
    inst, acts = random_starts(S, 6, 6, 2, 515)
    rows = []
    for tm in TENURES_MACH:
        for ti in TENURES_INS:
            t, out = wall(lambda: search.tabu_search(inst, acts, iterations=iterations, tenure_mach=tm, tenure_ins=ti))
            rows.append({"tenure_mach": tm, "tenure_ins": ti, "mean_best_objective": float(out["objective"].mean()),
                         "wall_s": t})
            print(json.dumps(rows[-1]), flush=True)
    best = min(rows, key=lambda r: r["mean_best_objective"])
    return {"instances": "device J6M6E2 seed 515", "S": S, "start": "random rollout", "iterations": iterations,
            "rows": rows, "best": best}


def replay_vs_materialised(S, J, M, E, K, flush):
    N = J * M
    inst, acts = random_starts(S, J, M, E, 91)
    env = fresh_env(inst, S, J, M, E)
    dev = env.device
    moves = search.neighbour_moves(acts, torch.as_tensor(inst["t"], device=dev), K, 1, 0)[:65536]
    R = int(moves.shape[0])
    src = torch.arange(S, device=dev)
    mv32 = moves.to(torch.int32)
    fused = lambda: env.replay_moves(acts, mv32)
    mater = lambda: env.replay(search.apply_moves(acts, moves), src[moves[:, 0]].to(torch.int32))
    a, b = fused(), mater()
    same = all(bool(torch.equal(x, y)) for x, y in zip(a, b))
    hashes = [[hashlib.sha256(x.cpu().numpy().tobytes()).hexdigest()[:16] for x in o] for o in (a, b)]
    for _ in range(2):
        fused()
        mater()
    tf = [ev_time(fused, flush) for _ in range(10)]
    tm = [ev_time(mater, flush) for _ in range(10)]
    f, m = float(np.median(tf)), float(np.median(tm))
    out = {"S": S, "J": J, "M": M, "E": E, "max_neighbours": K, "candidates": R, "replay_moves_s": f,
           "replay_moves_s_runs": tf, "materialised_s": m, "materialised_s_runs": tm, "materialised_over_replay_moves": m / f,
           "neighbour_bytes_materialised": 2 * R * N * 8, "move_bytes_replay_moves": R * 16,
           "outputs_equal": same, "hash_replay_moves": hashes[0], "hash_materialised": hashes[1],
           "all_valid": bool((a[2] == -1).all())}
    env.close()
    return out


def mip_dict(c):
    return {"Makespan": c[:, 0], "MachineEC": c[:, 1], "TransEC": c[:, 2], "MachineIdleT": c[:, 3]}


def starts():
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    out = []
    for tag in ("iotj", "n12800"):
        sd_op, sd_m = val.load_actor_state_dicts(g, tag)
        ja, ma = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")
        gr = val.greedy_validate(ja, ma, inst, return_actions=True)
        out.append(("greedy %s tf32" % tag, gr["actions"], True))
        bm = val.beam_validate(ja, ma, inst, 32, return_actions=True)
        out.append(("beam W=32 %s tf32" % tag, bm["best_actions"], True))
    env = envm.BatchedMTFJSPEnv(100, 6, 6, 2, left_shift=False, obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(W), (100, 1)))
    out.append(("GREEDY_R", rules.greedy_reward_rollout(env).cpu().numpy(), False))
    env.close()
    return inst, out


def quality(inst, start_list, tm, ti):
    mip = mip_dict(np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv13"])
    rows = []
    for name, acts, ls_on in start_list:
        t_ls, ls = wall(lambda: search.local_search(inst, acts, left_shift=ls_on, rounds=200))
        row = {"start": name, "left_shift": ls_on, "mean_objective_start": float(ls["history"][0].mean()),
               "local_search": {"mean_objective": float(ls["objective"].mean()),
                                "mean_mip_gap": float(val.mip_gaps(ls["final4"], mip)[1].mean()),
                                "rounds": int(ls["accepted"].shape[0]), "wall_s": t_ls, "replays": int(ls["replays"])},
               "tabu": []}
        for it in (200, 1000):
            t, tb = wall(lambda: search.tabu_search(inst, acts, left_shift=ls_on, iterations=it, tenure_mach=tm,
                                                    tenure_ins=ti))
            assert (tb["objective"] <= ls["objective"]).all(), name
            row["tabu"].append({"iterations": it, "mean_objective": float(tb["objective"].mean()),
                                "mean_mip_gap": float(val.mip_gaps(tb["final4"], mip)[1].mean()),
                                "better_than_local_search": int((tb["objective"] < ls["objective"]).sum()),
                                "wall_s": t, "replays": int(tb["replays"])})
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def split(inst, acts, tm, ti, first=100, last=200):
    """Per-part device time of iterations first .. last-1, replaying tabu_search's loop with events between parts."""
    S, N, M = inst["t"].shape
    env = fresh_env(inst, S, N // M, M, inst["edge"].shape[1])
    dev = env.device
    cur = torch.as_tensor(acts, device=dev, dtype=torch.int32)
    f4, _, _ = env.replay(cur)
    st = search.tabu_state(cur.transpose(0, 1).contiguous(), f4, W, M)
    t_dev = torch.as_tensor(inst["t"], device=dev)
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    parts = {"neighbour_moves": [], "replay_moves": [], "decision": []}
    cands, kinds, seen = [], [], []
    for it in range(last):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        base = st["cur"].transpose(0, 1)
        ev[0].record()
        moves = search.neighbour_moves(base, t_dev, None, 0, it)
        ev[1].record()
        mf4, _, _ = env.replay_moves(base, moves)
        ev[2].record()
        seg = torch.cat((zero, torch.cumsum(torch.bincount(moves[:, 0], minlength=S), 0)))
        ch = search.tabu_move(st, moves, seg, val._objective(mf4, W), mf4, it, tm, ti)
        ev[3].record()
        ev[3].synchronize()
        if it >= first:
            for k, (a, b) in zip(parts, zip(ev[:3], ev[1:])):
                parts[k].append(a.elapsed_time(b) * 1e-3)
            cands.append(int(moves.shape[0]))
            kinds.append(moves[ch.clamp(min=0).long(), 1][ch >= 0].cpu())
            seen.append(st["cur_obj"].cpu())
    env.close()
    med = {k: float(np.median(v)) for k, v in parts.items()}
    tot = sum(med.values())
    return {"S": S, "iterations": [first, last], "median_candidates": float(np.median(cands)),
            "median_s": med, "share": {k: v / tot for k, v in med.items()},
            "reassignment_share_of_moves_taken": float((torch.cat(kinds) == search.REASSIGN).double().mean()),
            "mean_distinct_current_objectives": float(np.mean([len(set(c.tolist())) for c in torch.stack(seen).t()]))}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "tabu_b200.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    res["tenure_sweep"] = tenure_sweep()
    if len(sys.argv) > 2 and sys.argv[2] == "sweep":
        print(json.dumps(res["tenure_sweep"]["best"]))
        return
    tm, ti = search.TENURE_MACH, search.TENURE_INS
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res["replay_moves"] = []
    for S, J, M, E, K in ((100, 6, 6, 2, None), (32, 10, 10, 3, None), (16, 30, 20, 5, 1024)):
        res["replay_moves"].append(replay_vs_materialised(S, J, M, E, K, flush))
        print(json.dumps(res["replay_moves"][-1]), flush=True)
    del flush
    torch.cuda.empty_cache()
    inst, start_list = starts()
    res["tenures_used"] = {"tenure_mach": tm, "tenure_ins": ti}
    res["shipped_100"] = quality(inst, start_list, tm, ti)
    res["iteration_split"] = split(inst, start_list[0][1], tm, ti)
    print(json.dumps(res["iteration_split"]), flush=True)
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(txt)


if __name__ == "__main__":
    main()
