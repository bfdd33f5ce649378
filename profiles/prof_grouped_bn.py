"""Per-instance BatchNorm groups on the tcgen05 job encoder and batched sampled validation (profiles/README.md,
"Grouped BatchNorm and best-of-K validation").  Settings that are compared run alternated in this one process.

  (a) greedy_validate of the 100 shipped J6M6E2 test instances with the shipped `iotj` checkpoint, both actors tf32:
      chunk=1 (100 batch-1 rollouts, the default) against chunk=100 (one batch, one BatchNorm group per instance);
      host clock around each whole call (it ends in a device synchronise), 3 alternated rounds.
  (b) one job-actor forward (tf32, scores of the candidates) at 65,536 J6M6 envs with groups=1 against groups=B;
      CUDA events, L2 overwritten (256 MB memset) before every timed call, median of 30 calls per setting, alternated.
  (c) sampled_validate at K = 1024 on the 100 instances (102,400 envs in chunks of 32,768): env-steps/s = K * 100 * 36
      over the wall time of the call (it ends in a device synchronise), after one untimed K = 64 warm-up.
  quality: mean best-of-K objective for K in {1, 16, 256, 1024}, the first K samples of the (c) run, tf32, next to the
      shipped CSV means of PPO-G (row 15), PPO-S (row 16) and MIP (row 13).
Prints the results as JSON and also writes them to the path given as the first argument, if any."""
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
GOLD = os.path.join(ROOT, "tests", "golden")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def objective(x):
    return 0.4 * x[..., 0] + 0.4 * (x[..., 1] + x[..., 3]) + 0.2 * x[..., 2]


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    res = {"gpu": gpu_info()}
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    job, mch = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")

    # (a)
    val.greedy_validate(job, mch, {k: v[:4] for k, v in inst.items()}, chunk=1)
    val.greedy_validate(job, mch, {k: v[:4] for k, v in inst.items()}, chunk=4)
    ta = {"chunk1_s": [], "chunk100_s": []}
    outs = {}
    for _ in range(3):
        for name, ch in (("chunk1_s", 1), ("chunk100_s", 100)):
            t, o = wall(lambda: val.greedy_validate(job, mch, inst, chunk=ch))
            ta[name].append(t)
            outs[name] = o["final4"]
    ta["final4_identical"] = bool((outs["chunk1_s"] == outs["chunk100_s"]).all())
    ta["csv15_same_chunk100"] = int((outs["chunk100_s"] == g["csv15"]).all(axis=1).sum())
    ta["speedup_median"] = float(np.median(ta["chunk1_s"]) / np.median(ta["chunk100_s"]))
    res["a_greedy_validate_100"] = ta

    # (b)
    B, J, M, E = 65536, 6, 6, 2
    d = ins.synthetic_instances(0, B, J, M, E, 5)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 5))
    env.obs(envm.MASK_ESA)
    for _ in range(5):
        env.random_step(seed=3)
    env.obs(envm.MASK_ESA)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def fwd(groups):
        with torch.no_grad():
            return job.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, None, env.job_mask, groups=groups,
                                return_logits=True)

    tb = {"groups1_ms": [], "groupsB_ms": []}
    for _ in range(3):
        fwd(1), fwd(B)
    for _ in range(30):
        for name, gr in (("groups1_ms", 1), ("groupsB_ms", B)):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fwd(gr)
            b.record()
            b.synchronize()
            tb[name].append(a.elapsed_time(b))
    res["b_job_forward_65536"] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
                                  for k, v in tb.items()}
    del env, flush
    torch.cuda.empty_cache()

    # (c) + quality
    val.sampled_validate(job, mch, inst, samples=64, seed=1)
    K = 1024
    t, o = wall(lambda: val.sampled_validate(job, mch, inst, samples=K, seed=2024))
    res["c_sampled_validate_K1024"] = {"seconds": t, "env_steps": K * 100 * 36, "env_steps_per_s": K * 100 * 36 / t}
    obj = o["objective"]
    s16 = np.load(os.path.join(GOLD, "sampled_golden.npz"))
    res["quality_tf32"] = {"best_of_%d" % k: float(obj[:k].min(axis=0).mean()) for k in (1, 16, 256, 1024)}
    res["quality_tf32"]["sample_mean"] = float(obj.mean())
    res["quality_csv"] = {"PPO-G_row15": float(objective(g["csv15"]).mean()), "PPO-S_row16": float(objective(s16["csv16"]).mean()),
                          "MIP_row13": float(objective(s16["csv13"]).mean())}
    txt = json.dumps(res, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        open(sys.argv[1], "w").write(txt)


if __name__ == "__main__":
    main()
