"""Before / after timing of the fused episode reset on workload A's random step (J6M6E2, 65,536 envs):
MTFJSP_FUSED_RESET=1 runs the reset inside the next step launch, =0 as reset_copy_kernel + scaler_kernel at the call.
Two envs, one per setting (the switch is read when an env is created), timed in turn, ROUNDS times: each turn is
bench.py's protocol -- K = 360 steps per timed region (episodes of 36 steps wrap inside it: reset + scaler reset
every 36 steps), median of 15 regions, CUDA events.  Reported per setting and round:
  ms_per_step      timed-region time / K
  step_kernel_us   mean of CUDA events around each random_step launch of steps 2..36 of an episode
  reset_us         events around [reset + scaler_reset + first step of the episode] minus step_kernel_us: what the
                   reset costs per episode
The card's name and power limit are read in the same process.  The JSON goes to the path given as the first
argument, if any."""
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

J, M, E, B, SEED = 6, 6, 2, 65536, 1002
N = J * M
K, REPEATS, ROUNDS = 360, 15, int(os.environ.get("ROUNDS", "5"))
SETTINGS = {"eager_reset": "0", "fused_reset": "1"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi failed: %r" % e
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def make(setting, d, w):
    os.environ["MTFJSP_FUSED_RESET"] = SETTINGS[setting]
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    return {"env": env, "s": 0}


def one_step(st, w):
    env = st["env"]
    if st["s"] == N:
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


def episode_split(st, w, episodes=3):
    """per-launch step time (steps 2..N) and the reset's cost per episode"""
    env = st["env"]
    steps, heads = [], []
    for _ in range(episodes):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(N)]
        ev[0][0].record()
        env.reset(w)
        env.scaler_reset()
        env.random_step(seed=1234, env_offset=0)
        ev[0][1].record()
        for s in range(1, N):
            ev[s][0].record()
            env.random_step(seed=1234, env_offset=0)
            ev[s][1].record()
        torch.cuda.synchronize()
        steps += [a.elapsed_time(b) for a, b in ev[1:]]
        heads.append(ev[0][0].elapsed_time(ev[0][1]))
    st["s"] = N
    step_us = 1e3 * statistics.mean(steps)
    return step_us, 1e3 * statistics.median(heads) - step_us


def main():
    torch.cuda.set_device(0)
    d = ins.synthetic_instances(0, B, J, M, E, SEED)
    w = torch.as_tensor(ins.random_weights(0, B, SEED)).cuda()
    envs = {k: make(k, d, w) for k in SETTINGS}
    for st in envs.values():  # warm-up: every launch shape, both directions, a reset
        for _ in range(2 * N):
            one_step(st, w)
    rows = []
    for r in range(ROUNDS):
        for k, st in envs.items():
            ms = timed_region(st, w)
            step_us, reset_us = episode_split(st, w)
            rows.append({"round": r, "setting": k, "ms_per_step": ms, "step_kernel_us": step_us, "reset_us": reset_us})
            print("round %d %-14s %.5f ms/step  step kernel %.2f us  reset %.1f us/episode" % (r, k, ms, step_us, reset_us),
                  flush=True)
    summary = {}
    for k in SETTINGS:
        xs = [x for x in rows if x["setting"] == k]
        ms = [x["ms_per_step"] for x in xs]
        summary[k] = {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms),
                      "spread": max(ms) - min(ms), "step_kernel_us_median": statistics.median(x["step_kernel_us"] for x in xs),
                      "reset_us_median": statistics.median(x["reset_us"] for x in xs),
                      "env_steps_per_s": B / (statistics.median(ms) * 1e-3)}
    old = summary["eager_reset"]["ms_per_step_median"]
    for k in SETTINGS:
        summary[k]["speedup_vs_eager"] = old / summary[k]["ms_per_step_median"]
    out = {"card": card(), "workload": "J6M6E2 %d envs, K=%d, median of %d regions, %d rounds" % (B, K, REPEATS, ROUNDS),
           "summary": summary, "rows": rows}
    print(json.dumps({"card": out["card"], "summary": summary}, indent=1))
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
