"""Pareto fronts over the three targets (profiles/README.md, "Pareto fronts and hypervolume").

  (a) mtfjsp_pareto_filter at S = 100 segments of P = 1,024 and 8,192 points each (mk and tt integer-valued, ec
      continuous, near a trade-off surface, so that a large share is non-dominated and ties are common): CUDA events
      around each call, median of 10 after 2 untimed calls.  Against a torch broadcast restatement of the same test in
      chunks of at most 2^25 (candidate, point) pairs; the two outputs are compared in the same run.
  (b) mtfjsp_hypervolume3 at S = 100 segments of n = 256 and 4,096 points on a plane (mutually non-dominated): events,
      median of 10.
  (c) Quality on the 100 shipped J6M6E2 test instances (tests/golden/pdr_golden.npz), tf32 actors of
      policy_golden.npz: hypervolume_table (one reference point per instance, 1.1 x the componentwise max over all
      methods) over greedy `iotj` and `n12800`, beam W = 32 `iotj` and `n12800` (all W finals), sampled K = 1,024 `iotj`,
      the union of 15 local_search runs under the weight vectors of the step-0.25 lattice on the simplex (each started
      from the sampled schedule that is best under its weights), and pareto_local_search started from the sampled front
      (defaults: expand 8, max_archive 256, 200 rounds), and again stopped after the rounds that match the lattice union's
      replay count at the first run's mean replays per round.  Wall time (host clock around work that ends in a
      synchronise) and replay counts of both searches, and on how many instances each method's front weakly dominates
      the MIP point (sampled_golden.npz row csv13).
Prints the results as JSON and writes them to the path given as the first argument (default profiles/pareto_b200.json)."""
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
    return torch.stack((torch.round(200 * w[:, 0]), 100 * w[:, 1], torch.round(50 * w[:, 2])), 1)


def torch_filter(obj, S, P, pairs=1 << 25):
    """The dominance test as torch broadcasts over equal-length segments: candidates in chunks against their segment."""
    o = obj.view(S, P, 3)
    fin = torch.isfinite(o).all(-1)
    q = torch.where(fin[..., None], o, float("inf"))
    idx = torch.arange(P, device=obj.device)
    keep = torch.empty((S, P), dtype=torch.bool, device=obj.device)
    cs = max(1, min(P, pairs // P))
    sg = max(1, pairs // (P * cs))
    for s0 in range(0, S, sg):
        for c0 in range(0, P, cs):
            pc = o[s0:s0 + sg, c0:c0 + cs]                                   # [g,c,3]
            qq = q[s0:s0 + sg]                                               # [g,P,3]
            le = (qq[:, None] <= pc[:, :, None]).all(-1)
            eq = (qq[:, None] == pc[:, :, None]).all(-1)
            dom = (le & (~eq | (idx[None, None, :] < idx[c0:c0 + cs, None]))).any(-1)
            keep[s0:s0 + sg, c0:c0 + cs] = ~dom & fin[s0:s0 + sg, c0:c0 + cs]
    return keep.view(-1)


def filter_timing(S, P):
    obj = points(S, P, 5 + P)
    seg = torch.arange(S + 1, dtype=torch.int64, device="cuda") * P
    k = pareto.pareto_filter(obj, seg, P)
    t_k, runs_k = ev_median(lambda: pareto.pareto_filter(obj, seg, P))
    kt = torch_filter(obj, S, P)
    t_t, runs_t = ev_median(lambda: torch_filter(obj, S, P), runs=3, warm=1)
    return {"S": S, "P_per_segment": P, "pairs": S * P * P, "kernel_s": t_k, "kernel_s_runs": runs_k, "torch_s": t_t,
            "torch_s_runs": runs_t, "speedup": t_t / t_k, "outputs_equal": bool(torch.equal(k, kt)),
            "kept_fraction": float(k.float().mean())}


def hv_timing(S, n):
    g = torch.Generator(device="cuda").manual_seed(77 + n)
    w = torch.rand((S * n, 3), generator=g, device="cuda", dtype=torch.float64)
    pts = (w / w.sum(1, keepdim=True) * torch.tensor([200.0, 100.0, 50.0], device="cuda", dtype=torch.float64)).contiguous()
    seg = torch.arange(S + 1, dtype=torch.int64, device="cuda") * n
    ref = torch.tensor(pareto.reference_point(pts.view(S, n, 3).transpose(0, 1).cpu().numpy()), device="cuda")
    t, runs = ev_median(lambda: pareto.hypervolume(pts, seg, ref))
    hv = pareto.hypervolume(pts, seg, ref).cpu().numpy()
    return {"S": S, "n": n, "points": "uniform on the simplex scaled by (200, 100, 50): mutually non-dominated",
            "kernel_s": t, "kernel_s_runs": runs, "mean_hypervolume": float(hv.mean())}


def lattice(step=0.25):
    k = int(round(1 / step))
    return [(a * step, b * step, (k - a - b) * step) for a in range(k + 1) for b in range(k + 1 - a)]


def quality():
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    S = inst["t"].shape[0]
    mip = np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv13"][:S]
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    sets, rows, acts = {}, {}, {}
    for tag in ("iotj", "n12800"):
        sd_op, sd_m = val.load_actor_state_dicts(g, tag)
        ja, ma = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")
        sets["greedy %s" % tag] = val.greedy_validate(ja, ma, inst)["final4"]
        sets["beam W=32 %s" % tag] = val.beam_validate(ja, ma, inst, 32)["final4"]
        if tag == "iotj":
            t, sp = wall(lambda: val.sampled_validate(ja, ma, inst, 1024, seed=0, return_actions=True))
            sets["sampled K=1024 iotj"] = sp["final4"]
            rows["sampled_wall_s"] = t
            acts = sp["actions"]                                               # [N,K,S,2]
    sf4 = sets["sampled K=1024 iotj"]
    cols = np.arange(S)
    # local search under every lattice weight vector, each from the sampled schedule best under those weights
    ls_f4, ls_t, ls_rep, ls_rows = [], 0.0, 0, []
    for w in lattice():
        best = np.argmin(val._objective(sf4, w), axis=0)
        t, out = wall(lambda: search.local_search(inst, acts[:, best, cols], weights=w, rounds=200))
        ls_f4.append(out["final4"])
        ls_t += t
        ls_rep += out["replays"]
        ls_rows.append({"weights": w, "rounds_run": int(out["accepted"].shape[0]), "wall_s": t, "replays": out["replays"],
                        "mean_objective_before": float(val._objective(sf4[best, cols], w).mean()),
                        "mean_objective_after": float(out["objective"].mean())})
        print(json.dumps(ls_rows[-1]), flush=True)
    sets["local_search lattice union"] = np.stack(ls_f4)
    fr = pareto.front(sf4)
    K = max(len(f) for f in fr)
    start = np.zeros((acts.shape[0], K, S, 2), dtype=np.int32)
    for s, f in enumerate(fr):                                               # pad with the front's first member
        start[:, :, s] = acts[:, np.r_[f, np.full(K - len(f), f[0])], s]
    t, pls = wall(lambda: search.pareto_local_search(inst, start))
    A = pls["final4"].shape[1]
    sets["pareto_local_search"] = pls["final4"].transpose(1, 0, 2)           # [A,S,4], NaN rows take no part
    # the same search stopped after the rounds that, at its mean replays per round, match the lattice union's replays
    r_eq = max(1, int(ls_rep * pls["truncated"].shape[0] / pls["replays"]))
    t_eq, pls_eq = wall(lambda: search.pareto_local_search(inst, start, rounds=r_eq))
    sets["pareto_local_search, lattice replay budget"] = pls_eq["final4"].transpose(1, 0, 2)
    tab = pareto.hypervolume_table(sets)
    mo = pareto.objectives(mip)
    dominated = {}
    for name, f4 in sets.items():
        o = pareto.objectives(f4 if f4.ndim == 3 else f4[None])              # [K,S,3]
        dominated[name] = int(sum(bool((o[:, s] <= mo[s]).all(-1).any()) for s in range(S)))
    res = {"instances": S, "methods": list(sets),
           "mean_hypervolume": {k: float(np.mean(v)) for k, v in tab["hypervolume"].items()},
           "mean_hypervolume_union": float(tab["union"].mean()),
           "instances_best_hypervolume": {k: int((v >= np.max(np.stack(list(tab["hypervolume"].values())), 0)).sum())
                                          for k, v in tab["hypervolume"].items()},
           "mip_point_weakly_dominated_on_instances": dominated,
           "mean_front_size": {k: float(np.mean([len(f) for f in pareto.front(v if v.ndim == 3 else v[None])]))
                               for k, v in sets.items() if not k.startswith("pareto_local_search")},
           "sampled_front_size_mean": float(np.mean([len(f) for f in fr])),
           "sampled_wall_s": rows["sampled_wall_s"],
           "local_search_lattice": {"runs": ls_rows, "wall_s": ls_t, "replays": ls_rep},
           "pareto_local_search": {"wall_s": t, "replays": int(pls["replays"]),
                                   "rounds_run": int(pls["truncated"].shape[0]),
                                   "instances_truncated": int(pls["truncated"].any(0).sum()),
                                   "mean_archive": float(pls["count"].mean()), "max_archive": A,
                                   "unexplored_left": int(sum((~pls["explored"][s, :pls["count"][s]]).sum()
                                                              for s in range(S))),
                                   "mean_hypervolume_own_ref_start": float(pls["hypervolume"][0].mean()),
                                   "mean_hypervolume_own_ref_end": float(pls["hypervolume"][-1].mean())},
           "pareto_local_search_lattice_budget": {"wall_s": t_eq, "replays": int(pls_eq["replays"]), "rounds_run": r_eq,
                                                  "mean_archive": float(pls_eq["count"].mean())}}
    print(json.dumps(res), flush=True)
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "pareto_b200.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    res["filter"] = []
    for P in (1024, 8192):
        res["filter"].append(filter_timing(100, P))
        print(json.dumps(res["filter"][-1]), flush=True)
    res["hypervolume"] = []
    for n in (256, 4096):
        res["hypervolume"].append(hv_timing(100, n))
        print(json.dumps(res["hypervolume"][-1]), flush=True)
    res["quality_shipped_100"] = quality()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
