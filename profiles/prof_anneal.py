"""Parallel tempering on the neighbour replay (profiles/README.md, "Parallel tempering").

  (a) Default sweep, run first: anneal_search (left shift on) on 64 device-generated J6M6E2 instances
      (instances.device_instances, seed 515) from random-rollout sequences, at about 7 M replays per cell, for
      K in {32, 128, 512} x t_max in {0.003, 0.01, 0.03, 0.1} x t_min in {1e-4, 1e-3} x swap_every in {1, 10}: mean
      best objective; tabu_search's defaults at 200 iterations on the same starts for scale.
  (b) On the 100 shipped J6M6E2 test instances, from the five starts of the tabu table (prof_tabu.starts), tabu_search
      at 200 and 1,000 iterations and anneal_search's defaults at the same replay counts: mean objective, mean
      validate.mip_gaps gap to the MIP row (csv13), instances strictly better / worse than tabu, wall time (host clock
      ending in a synchronise).
  (c) 32 device-generated J10M10E3 and 16 J30M20E5 instances from random-rollout sequences: anneal_search against
      tabu_search at equal replays (full neighbourhood at J10M10, max_neighbours=1024 at J30M20) and local_search.
  (d) One iteration's device time split into anneal_propose, replay_moves and objective + anneal_step (CUDA events,
      medians over iterations 100 .. 199 on the shipped instances from greedy `iotj`), and chains proposed per second.
  (e) `sass PARENT_LIB`: no GPU; -Xptxas -v of mtfjsp_anneal.cu and a per-Function comparison of `cuobjdump -sass` of
      the in-tree library against PARENT_LIB (the parent commit's build), merged into the output JSON.
Prints the results as JSON and writes them to the path given as the first argument (default profiles/anneal_b200.json);
a second argument `sweep` stops after (a)."""
import importlib
import json
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import prof_tabu as pt  # noqa: E402  (the start builders and gpu_info of the tabu profile)

val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
GOLD = os.path.join(ROOT, "tests", "golden")
W = (0.4, 0.4, 0.2)
KS, T_MAXS, T_MINS, SWAPS = (32, 128, 512), (0.003, 0.01, 0.03, 0.1), (1e-4, 1e-3), (1, 10)
SWEEP_REPLAYS = 7_000_000


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def iterations_for(replays, S, K):
    """anneal_search iterations whose replays (the start included) come closest to `replays`."""
    return max(1, int(round((replays - S) / (S * K))))


def sweep(S=64):
    inst, acts = pt.random_starts(S, 6, 6, 2, 515)
    rows = []
    for K in KS:
        its = iterations_for(SWEEP_REPLAYS, S, K)
        for t_max in T_MAXS:
            for t_min in T_MINS:
                for se in SWAPS:
                    lad = search.anneal_ladder(K, t_max, t_min)
                    t, out = wall(lambda: search.anneal_search(inst, acts, iterations=its, ladder=lad, swap_every=se))
                    rows.append({"K": K, "t_max": t_max, "t_min": t_min, "swap_every": se, "iterations": its,
                                 "replays": int(out["replays"]), "mean_best_objective": float(out["objective"].mean()),
                                 "accept_rate_coldest_hottest": [float(out["accept_rate"][0]),
                                                                 float(out["accept_rate"][-1])],
                                 "mean_swap_rate": float(np.nanmean(out["swap_rate"])), "wall_s": t})
                    print(json.dumps(rows[-1]), flush=True)
    best = min(rows, key=lambda r: r["mean_best_objective"])
    # K = 32, the least K of the grid, won it: fewer chains beyond the grid at the winner's temperatures
    beyond = []
    for K in (8, 16):
        its = iterations_for(SWEEP_REPLAYS, S, K)
        lad = search.anneal_ladder(K, best["t_max"], best["t_min"])
        t, out = wall(lambda: search.anneal_search(inst, acts, iterations=its, ladder=lad, swap_every=best["swap_every"]))
        beyond.append({"K": K, "iterations": its, "replays": int(out["replays"]),
                       "mean_best_objective": float(out["objective"].mean()), "wall_s": t})
        print(json.dumps(beyond[-1]), flush=True)
    t, tb = wall(lambda: search.tabu_search(inst, acts, iterations=200))
    return {"instances": "device J6M6E2 seed 515", "S": S, "start": "random rollout",
            "mean_start_objective": float(tb["history"][0].mean()), "rows": rows, "best": best, "beyond_grid": beyond,
            "tabu_200": {"mean_objective": float(tb["objective"].mean()), "replays": int(tb["replays"]), "wall_s": t}}


def shipped(inst, start_list):
    mip = pt.mip_dict(np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv13"])
    S = inst["t"].shape[0]
    K = search.ANNEAL_CHAINS
    rows = []
    for name, acts, ls_on in start_list:
        row = {"start": name, "left_shift": ls_on, "budgets": []}
        for it in (200, 1000):
            t_tb, tb = wall(lambda: search.tabu_search(inst, acts, left_shift=ls_on, iterations=it))
            ai = iterations_for(tb["replays"], S, K)
            t_an, an = wall(lambda: search.anneal_search(inst, acts, left_shift=ls_on, iterations=ai))
            row["mean_objective_start"] = float(tb["history"][0].mean())
            row["budgets"].append({
                "tabu": {"iterations": it, "mean_objective": float(tb["objective"].mean()),
                         "mean_mip_gap": float(val.mip_gaps(tb["final4"], mip)[1].mean()), "wall_s": t_tb,
                         "replays": int(tb["replays"])},
                "anneal": {"iterations": ai, "mean_objective": float(an["objective"].mean()),
                           "mean_mip_gap": float(val.mip_gaps(an["final4"], mip)[1].mean()), "wall_s": t_an,
                           "replays": int(an["replays"]), "better_than_tabu": int((an["objective"] < tb["objective"]).sum()),
                           "worse_than_tabu": int((an["objective"] > tb["objective"]).sum()),
                           "accept_rate_coldest_hottest": [float(an["accept_rate"][0]), float(an["accept_rate"][-1])]}})
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def larger():
    out = []
    for S, J, M, E, K_nb, tabu_its, ls_rounds in ((32, 10, 10, 3, None, 100, 200), (16, 30, 20, 5, 1024, 30, 30)):
        inst, acts = pt.random_starts(S, J, M, E, 91)
        t_ls, ls = wall(lambda: search.local_search(inst, acts, rounds=ls_rounds, max_neighbours=K_nb))
        t_tb, tb = wall(lambda: search.tabu_search(inst, acts, iterations=tabu_its, max_neighbours=K_nb))
        ai = iterations_for(tb["replays"], S, search.ANNEAL_CHAINS)
        t_an, an = wall(lambda: search.anneal_search(inst, acts, iterations=ai))
        row = {"S": S, "J": J, "M": M, "E": E, "max_neighbours": K_nb,
               "mean_objective_start": float(ls["history"][0].mean()),
               "local_search": {"rounds": int(ls["accepted"].shape[0]), "mean_objective": float(ls["objective"].mean()),
                                "wall_s": t_ls, "replays": int(ls["replays"])},
               "tabu": {"iterations": tabu_its, "mean_objective": float(tb["objective"].mean()), "wall_s": t_tb,
                        "replays": int(tb["replays"])},
               "anneal": {"iterations": ai, "mean_objective": float(an["objective"].mean()), "wall_s": t_an,
                          "replays": int(an["replays"]), "better_than_tabu": int((an["objective"] < tb["objective"]).sum()),
                          "worse_than_tabu": int((an["objective"] > tb["objective"]).sum())}}
        print(json.dumps(row), flush=True)
        out.append(row)
    return out


def split(inst, acts, first=100, last=200):
    """Per-part device time of iterations first .. last-1, replaying anneal_search's loop with events between parts."""
    S, N, M = inst["t"].shape
    K = search.ANNEAL_CHAINS
    env = pt.fresh_env(inst, S, N // M, M, inst["edge"].shape[1])
    dev = env.device
    cur = torch.as_tensor(acts, device=dev, dtype=torch.int32)
    f4, _, _ = env.replay(cur)
    st = search.anneal_state(cur.transpose(0, 1).contiguous(), f4, W, K)
    temp = torch.as_tensor(search.anneal_ladder(), device=dev)[None, :] * st["best_obj"][:, None]
    t_dev = torch.as_tensor(inst["t"], device=dev, dtype=torch.float64)
    src = torch.arange(S * K, dtype=torch.int32, device=dev) // K
    parts = {"propose": [], "replay_moves": [], "objective_and_step": []}
    for it in range(last):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        moves = search.anneal_propose(t_dev, st["cur"], 0, it)
        ev[1].record()
        mf4, _, fi = env.replay_moves(st["cur"].transpose(0, 1), moves, src)
        ev[2].record()
        search.anneal_step(st, moves, fi, val._objective(mf4, W), mf4, temp, 0, it, search._swap_parity(it, 1), M)
        ev[3].record()
        ev[3].synchronize()
        if it >= first:
            for k, (a, b) in zip(parts, zip(ev[:3], ev[1:])):
                parts[k].append(a.elapsed_time(b) * 1e-3)
    env.close()
    med = {k: float(np.median(v)) for k, v in parts.items()}
    tot = sum(med.values())
    return {"S": S, "K": K, "chains": S * K, "iterations": [first, last], "median_s": med,
            "share": {k: v / tot for k, v in med.items()}, "chains_per_s": S * K / tot}


def _sass_functions(lib_path):
    txt = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None and "/*" in line:  # instructions and their encodings, not the next file's header
            funcs[name].append(line)
    # anonymous-namespace names carry a hash of the build path: compare them without it
    anon = re.compile(r"\d+_GLOBAL__N__[0-9a-f]{8}_\d+_(\w+?)_cu_[0-9a-f]{8}")
    return {anon.sub(r"_GLOBAL__N_\1", k): anon.sub(r"_GLOBAL__N_\1", "\n".join(v)) for k, v in funcs.items()}


def compiler(parent_lib):
    src = os.path.join(libm.SRC_DIR, "mtfjsp_anneal.cu")
    cmd = ["nvcc"] + libm.NVCC_FLAGS + libm.EXTRA_FLAGS["mtfjsp_anneal.cu"] + ["-Xptxas", "-v", "-c", "-o", os.devnull,
                                                                              src]
    log = subprocess.run(cmd, capture_output=True, text=True, check=True).stderr
    ptxas = {}
    for fn, body in re.findall(r"Function properties for (\S+)\n(.*?)(?=ptxas info    : Compiling|\Z)", log, re.S):
        kern = re.search(r"(anneal_(?:step|propose)_kernel)", fn).group(1)
        ptxas[kern] = " ".join(x.strip() for x in body.strip().splitlines() if "Compile time" not in x)
    new, old = _sass_functions(libm.LIB_PATH), _sass_functions(parent_lib)
    changed = sorted(k for k in old if new.get(k) != old[k])
    return {"ptxas": ptxas, "parent_functions": len(old), "functions": len(new),
            "parent_functions_changed_or_missing": changed, "added": sorted(set(new) - set(old))}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "anneal_b200.json")
    if len(sys.argv) > 3 and sys.argv[2] == "sass":
        res = json.load(open(out_path)) if os.path.exists(out_path) else {}
        res["compiler"] = compiler(sys.argv[3])
        print(json.dumps(res["compiler"], indent=1))
        with open(out_path, "w") as f:
            f.write(json.dumps(res, indent=1))
        return
    torch.cuda.set_device(0)
    res = {"gpu": pt.gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    res["sweep"] = sweep()
    print(json.dumps(res["sweep"]["best"]), flush=True)
    if len(sys.argv) > 2 and sys.argv[2] == "sweep":
        res["gpu_after"] = pt.gpu_info()
    else:
        res["defaults"] = {"K": search.ANNEAL_CHAINS, "t_max": search.ANNEAL_T_MAX, "t_min": search.ANNEAL_T_MIN,
                           "swap_every": search.ANNEAL_SWAP_EVERY}
        inst, start_list = pt.starts()
        res["shipped_100"] = shipped(inst, start_list)
        res["larger"] = larger()
        res["iteration_split"] = split(inst, start_list[0][1])
        print(json.dumps(res["iteration_split"]), flush=True)
        res["gpu_after"] = pt.gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
