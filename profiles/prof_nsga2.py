"""NSGA-II on the device (profiles/README.md, "NSGA-II").

  (a) mtfjsp_pareto_rank at S = 100 segments of P = 512 and 4,096 points each (the point cloud of prof_pareto.py: mk
      and tt integer-valued, ec continuous, around a trade-off surface, so ties are common and there are many fronts):
      CUDA events around each call, median of 10 after 2 untimed calls.  Against a torch restatement that peels fronts
      with repeated mtfjsp_pareto_filter calls (one host read per front); the two outputs are compared in the same run.
  (b) mtfjsp_offspring on 65,536 J6M6E2, 16,384 J10M10E2 and 4,096 J30M20E5 children of 1,024 random parents of 64
      device-generated instances (p_swap 0.2, p_mach 1/N), and as many random children: events, median of 10.
  (c) Quality on the 100 shipped J6M6E2 test instances (tests/golden/pdr_golden.npz), tf32 `iotj` actors of
      policy_golden.npz: hypervolume_table (one reference point per instance over all methods) over sampled K = 1,024,
      pareto_local_search from the sampled front at 44 and 200 rounds (defaults otherwise), nsga2 (pop 256, defaults)
      from the sampled front and from random individuals only, for 100 generations and again for the generations whose
      replays match each local-search run's.  Wall time (host clock around work that ends in a synchronise), replays,
      and on how many instances each front weakly dominates the MIP point (sampled_golden.npz row csv13).
  (d) One nsga2 run from random individuals at J30M20E5 on 128 device-generated instances.
  (e) Where a generation's time goes, at the sizes of (c) from random individuals (100 instances, pop 256): the wall
      time per generation (a 200-generation run minus a 0-generation run, over 200), against the stream time (CUDA
      events, median of 10) of each step alone at one generation's sizes: the 25,600 children's replay, the offspring
      launch, the selection (rank, crowding distance and sorts of 512 members per instance) and the front-0
      hypervolume.
Prints the results as JSON and writes them to the path given as the first argument (default profiles/nsga2_b200.json)."""
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
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
pareto = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.pareto")
evolve = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.evolve")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
GOLD = os.path.join(ROOT, "tests", "golden")


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


def ev_median(fn, runs=10, warm=2):
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
    return float(np.median(ts)), ts


def points(S, P, seed):
    """[S*P,3]: mk and tt integers, ec continuous, scattered around mk/200 + ec/100 + tt/50 = 3."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = torch.rand((S * P, 3), generator=g, device="cuda", dtype=torch.float64)
    w = w / w.sum(1, keepdim=True) * (3.0 + 0.3 * torch.rand((S * P, 1), generator=g, device="cuda", dtype=torch.float64))
    return torch.stack((torch.round(200 * w[:, 0]), 100 * w[:, 1], torch.round(50 * w[:, 2])), 1).contiguous()


def torch_rank(obj, seg, P):
    """Non-dominated sorting by peeling: the filter's front of the points not yet ranked, one front per call."""
    rank = torch.full((obj.shape[0],), np.iinfo(np.int32).max, dtype=torch.int32, device=obj.device)
    left = torch.isfinite(obj).all(1)
    f = 0
    while bool(left.any()):
        keep = pareto.pareto_filter(torch.where(left[:, None], obj, float("nan")), seg, P)
        rank[keep] = f
        left &= ~keep
        f += 1
    return rank


def rank_timing(S, P):
    obj = points(S, P, 5 + P)
    seg = torch.arange(S + 1, dtype=torch.int64, device="cuda") * P
    r = pareto.pareto_rank(obj, seg, P)
    t_k, runs_k = ev_median(lambda: pareto.pareto_rank(obj, seg, P))
    rt = torch_rank(obj, seg, P)
    t_t, runs_t = ev_median(lambda: torch_rank(obj, seg, P), runs=3, warm=1)
    return {"S": S, "P_per_segment": P, "kernel_s": t_k, "kernel_s_runs": runs_k, "torch_peel_s": t_t,
            "torch_peel_s_runs": runs_t, "speedup": t_t / t_k, "outputs_equal": bool(torch.equal(r, rt)),
            "fronts_max": int(r.max()) + 1, "front0_fraction": float((r == 0).float().mean())}


def offspring_timing(J, M, E, C, S=64, P=1024):
    d = ins.device_instances(0, S, J, M, E, seed=3)
    t = d["t"].contiguous()
    N = J * M
    inst_p = torch.arange(P, device="cuda", dtype=torch.int32) % S
    par = evolve._offspring_flat(t, M, torch.zeros((0, N, 2), dtype=torch.int32, device="cuda"),
                                 torch.full((P, 2), -1, dtype=torch.int32, device="cuda"), inst_p, 1, 0.0, 0.0)
    g = torch.Generator(device="cuda").manual_seed(C)
    k = torch.randint(0, P // S, (C, 2), generator=g, device="cuda", dtype=torch.int32)
    inst = torch.randint(0, S, (C,), generator=g, device="cuda", dtype=torch.int32)
    pair = (k * S + inst[:, None]).contiguous()                              # parents of the child's instance
    rnd = torch.full((C, 2), -1, dtype=torch.int32, device="cuda")
    x = lambda: evolve._offspring_flat(t, M, par, pair, inst, 7, 0.2, 1.0 / N)
    r = lambda: evolve._offspring_flat(t, M, par, rnd, inst, 7, 0.0, 0.0)
    t_x, runs_x = ev_median(x)
    t_r, runs_r = ev_median(r)
    kids = x()
    assert bool((kids >= 0).all())
    return {"size": "J%dM%dE%d" % (J, M, E), "children": C, "parents": P, "crossover_s": t_x, "crossover_s_runs": runs_x,
            "random_s": t_r, "random_s_runs": runs_r, "children_per_s_crossover": C / t_x,
            "children_per_s_random": C / t_r}


def quality():
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    S = inst["t"].shape[0]
    mip = np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv13"][:S]
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    ja, ma = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")
    t_s, sp = wall(lambda: val.sampled_validate(ja, ma, inst, 1024, seed=0, return_actions=True))
    acts = sp["actions"]                                                     # [N,K,S,2]
    sets = {"sampled K=1024 iotj": sp["final4"]}
    runs = {"sampled K=1024 iotj": {"wall_s": t_s, "replays": None}}
    fr = pareto.front(sp["final4"])
    K = max(len(f) for f in fr)
    start = np.zeros((acts.shape[0], K, S, 2), dtype=np.int32)
    for s, f in enumerate(fr):                                               # pad with the front's first member
        start[:, :, s] = acts[:, np.r_[f, np.full(K - len(f), f[0])], s]
    budgets = {}
    for rounds in (44, 200):
        t, out = wall(lambda: search.pareto_local_search(inst, start, rounds=rounds))
        name = "pareto_local_search %d rounds" % rounds
        sets[name] = out["final4"].transpose(1, 0, 2)                        # [A,S,4], NaN rows take no part
        runs[name] = {"wall_s": t, "replays": int(out["replays"]), "rounds_run": int(out["truncated"].shape[0])}
        budgets[rounds] = int(out["replays"])
        print(json.dumps({name: runs[name]}), flush=True)
    pop = 256
    plans = [("sampled front", start, 100), ("random", None, 100)]
    for rounds, rep in budgets.items():
        plans.append(("sampled front", start, max(1, round((rep - S * K) / (S * pop)))))
        plans.append(("random", None, max(1, round((rep - S * pop) / (S * pop)))))
    for label, st, gens in plans:
        t, out = wall(lambda: evolve.nsga2(inst, st, pop=pop, generations=gens))
        name = "nsga2 from %s, %d generations" % (label, gens)
        o = out["final4"].transpose(1, 0, 2).copy()
        o[(out["rank"] != 0).T] = np.nan                                     # the rank-0 members only
        sets[name] = o
        runs[name] = {"wall_s": t, "replays": int(out["replays"]), "generations": gens, "pop": pop,
                      "mean_front0": float((out["rank"] == 0).sum(1).mean()),
                      "mean_hypervolume_own_ref_start": float(out["hypervolume"][0].mean()),
                      "mean_hypervolume_own_ref_end": float(out["hypervolume"][-1].mean())}
        print(json.dumps({name: runs[name]}), flush=True)
    tab = pareto.hypervolume_table(sets)
    mo = pareto.objectives(mip)
    dominated = {}
    for name, f4 in sets.items():
        o = pareto.objectives(f4)                                            # [K,S,3]
        dominated[name] = int(sum(bool((o[:, s] <= mo[s]).all(-1).any()) for s in range(S)))
    hvs = np.stack(list(tab["hypervolume"].values()))
    res = {"instances": S, "methods": list(sets), "runs": runs,
           "mean_hypervolume": {k: float(np.mean(v)) for k, v in tab["hypervolume"].items()},
           "mean_hypervolume_union": float(tab["union"].mean()),
           "instances_best_hypervolume": {k: int((v >= hvs.max(0)).sum()) for k, v in tab["hypervolume"].items()},
           "mip_point_weakly_dominated_on_instances": dominated}
    print(json.dumps(res), flush=True)
    return res


def large(S=128, pop=64, generations=50):
    d = {k: v.cpu().numpy() for k, v in ins.device_instances(0, S, 30, 20, 5, seed=11).items()}
    t, out = wall(lambda: evolve.nsga2(d, None, pop=pop, generations=generations))
    h = out["hypervolume"]
    return {"size": "J30M20E5", "instances": S, "pop": pop, "generations": generations, "wall_s": t,
            "replays": int(out["replays"]), "replays_per_s": out["replays"] / t,
            "mean_hypervolume_own_ref_start": float(h[0].mean()), "mean_hypervolume_own_ref_end": float(h[-1].mean()),
            "mean_front0": float((out["rank"] == 0).sum(1).mean())}


def breakdown(pop=256, generations=200):
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    S, N, M = inst["t"].shape
    t0, _ = wall(lambda: evolve.nsga2(inst, None, pop=pop, generations=0))
    tg, out = wall(lambda: evolve.nsga2(inst, None, pop=pop, generations=generations))
    env = evolve.BatchedMTFJSPEnv(S, N // M, M, inst["edge"].shape[1], left_shift=True, obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (S, 1)))
    dev = env.device
    t_dev = torch.as_tensor(inst["t"], device=dev)
    par = torch.as_tensor(out["actions"], device=dev).permute(1, 2, 0, 3).reshape(S * pop, N, 2).contiguous()
    inst_c = torch.arange(S, device=dev, dtype=torch.int32).repeat_interleave(pop)
    g = torch.Generator(device="cuda").manual_seed(1)
    pair = (inst_c[:, None] * pop + torch.randint(0, pop, (S * pop, 2), generator=g, device=dev, dtype=torch.int32))
    pair = pair.to(torch.int32).contiguous()
    kids = evolve._offspring_flat(t_dev, M, par, pair, inst_c, 5, 0.2, 1.0 / N)
    t_off, _ = ev_median(lambda: evolve._offspring_flat(t_dev, M, par, pair, inst_c, 5, 0.2, 1.0 / N))
    t_rep, _ = ev_median(lambda: search._replay_all(env, S * pop, lambda a, b: kids[a:b].transpose(0, 1), inst_c, 65536))
    f4k, _ = search._replay_all(env, S * pop, lambda a, b: kids[a:b].transpose(0, 1), inst_c, 65536)
    f4 = torch.cat((torch.as_tensor(out["final4"], device=dev), f4k.view(S, pop, 4)), 1)
    t_sel, _ = ev_median(lambda: evolve._select(f4, pop))
    ref = torch.as_tensor(out["ref"], device=dev)
    seg = torch.arange(S + 1, dtype=torch.int64, device=dev) * pop
    o = pareto.objectives(torch.as_tensor(out["final4"], device=dev)).reshape(S * pop, 3)
    t_hv, _ = ev_median(lambda: pareto.hypervolume(o, seg, ref))
    env.close()
    per_gen = (tg - t0) / generations
    return {"instances": S, "pop": pop, "generations": generations, "wall_s_per_generation": per_gen,
            "replay_children_s": t_rep, "offspring_s": t_off, "select_s": t_sel, "front_hypervolume_s": t_hv,
            "steps_sum_s": t_rep + t_off + t_sel + t_hv, "replay_share_of_generation": t_rep / per_gen}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "nsga2_b200.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    res["rank"] = []
    for P in (512, 4096):
        res["rank"].append(rank_timing(100, P))
        print(json.dumps(res["rank"][-1]), flush=True)
    res["offspring"] = []
    for J, M, E, C in ((6, 6, 2, 65536), (10, 10, 2, 16384), (30, 20, 5, 4096)):
        res["offspring"].append(offspring_timing(J, M, E, C))
        print(json.dumps(res["offspring"][-1]), flush=True)
    res["quality_shipped_100"] = quality()
    res["generation_breakdown"] = breakdown()
    print(json.dumps(res["generation_breakdown"]), flush=True)
    res["j30m20"] = large()
    print(json.dumps(res["j30m20"]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
