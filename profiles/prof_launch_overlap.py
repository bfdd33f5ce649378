"""Before / after timing of overlapped step launches on the random step: MTFJSP_LAUNCH_OVERLAP=1 lets a whole-batch
step launch start while the previous one finishes (programmatic dependent launch, per-warp completion epochs),
=0 keeps plain stream order.  Two envs, one per setting (the switch is read when an env is created), timed in turn,
ROUNDS times: each turn is bench.py's protocol -- K = 360 steps per timed region (episodes wrap inside it: reset +
scaler reset every N steps), median of 15 regions, CUDA events.  Reported per setting and round: ms_per_step
(timed-region time / K); per setting: median, min, max and spread over the rounds.
Usage: prof_launch_overlap.py [A|B|C] [out.json]  (bench.py's workloads; default A).  The card's name and power limit
are read in the same process."""
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")

WORKLOADS = {"A": (6, 6, 2, 65536, 1002), "B": (10, 10, 3, 16384, 1003), "C": (30, 20, 5, 4096, 1004)}
K, REPEATS, ROUNDS = 360, 15, int(os.environ.get("ROUNDS", "5"))
SETTINGS = {"stream_order": "0", "overlap": "1"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi failed: %r" % e
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def make(setting, wl, d, w):
    J, M, E, B, _ = wl
    os.environ["MTFJSP_LAUNCH_OVERLAP"] = SETTINGS[setting]
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    return {"env": env, "s": 0}


def one_step(st, w):
    env = st["env"]
    if st["s"] == env.N:
        env.reset(w)
        env.scaler_reset()
        st["s"] = 0
    env.random_step(seed=1234, env_offset=0)
    st["s"] += 1


def timed_region(st, w):
    times = []
    for _ in range(REPEATS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            one_step(st, w)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times) / K


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "A"
    wl = WORKLOADS[name]
    J, M, E, B, seed = wl
    torch.cuda.set_device(0)
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    w = torch.as_tensor(ins.random_weights(0, B, seed)).cuda()
    envs = {k: make(k, wl, d, w) for k in SETTINGS}
    for st in envs.values():  # warm-up: every launch shape, both directions, a reset
        for _ in range(2 * J * M):
            one_step(st, w)
    rows = []
    for r in range(ROUNDS):
        for k, st in envs.items():
            ms = timed_region(st, w)
            rows.append({"round": r, "setting": k, "ms_per_step": ms})
            print("%s round %d %-13s %.5f ms/step" % (name, r, k, ms), flush=True)
    for st in envs.values():
        assert st["env"].launch_overlap_error == 0
    summary = {}
    for k in SETTINGS:
        ms = [x["ms_per_step"] for x in rows if x["setting"] == k]
        summary[k] = {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms),
                      "spread": max(ms) - min(ms), "env_steps_per_s": B / (statistics.median(ms) * 1e-3)}
    summary["overlap"]["speedup"] = summary["stream_order"]["ms_per_step_median"] / summary["overlap"]["ms_per_step_median"]
    out = {"card": card(), "workload": "%s: J%dM%dE%d %d envs, K=%d, median of %d regions, %d rounds" % (
        name, J, M, E, B, K, REPEATS, ROUNDS), "summary": summary, "rows": rows}
    print(json.dumps({"card": out["card"], "workload": out["workload"], "summary": summary}, indent=1))
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
