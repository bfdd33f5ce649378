"""Env gather and beam-search validation (profiles/README.md, "Env gather and beam search").

  (a) mtfjsp_gather alone (the C entry point, not the torch copies of gather_from) at 4,096 and 65,536 J6M6E2 envs and
      4,096 J30M20E5 envs, idx a random permutation: CUDA events around each call, L2 overwritten (256 MB memset) before
      every timed call, median of 20 calls after 3 untimed ones; bytes = mtfjsp_bytes_per_gather (every copied record
      read once and written once) x envs.  Also gather_from whole (ABI call + index copies of the owned buffers).
  (b) beam_validate of the 100 shipped J6M6E2 test instances with the shipped `iotj` and `n12800` checkpoints, tf32 and
      fp32, W in {1, 2, 4, 8, 16, 32}: host clock around the whole call (it ends in a device synchronise), median of 3
      calls after one untimed call of the same W (env batches, library algorithm choices); per step = total / 36.
  (c) where a beam step goes: torch.profiler (CPU and CUDA activities) around one W = 4 beam_validate call (tf32,
      `iotj`, 100 instances, after an untimed one), with host ranges around each stage of the step (job actor, candidate
      machine features, machine actor, selection, gather_from, env step); host time per stage, device time per kernel
      (the library's kernels are launched through ctypes, so the profiler does not attribute them to a stage).
      A run of its own: tracing slows the host, so (b) is the end-to-end figure.
  quality: mean over the 100 instances of the best objective for each W, next to greedy_validate and to the best of
      K = W samples of sampled_validate (seed 0), which runs the same number of env-steps (K x 36 per instance).
Prints the results as JSON and writes them to the path given as the first argument (default profiles/beam_b200.json)."""
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
GOLD = os.path.join(ROOT, "tests", "golden")
WIDTHS = (1, 2, 4, 8, 16, 32)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def env_pair(B, J, M, E):
    d = ins.synthetic_instances(0, B, J, M, E, 99)
    src = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    src.load(d["t"], d["p"], d["transT"], d["edge"])
    src.scaler_init()
    src.reset(ins.random_weights(0, B, 99))
    src.obs()
    for _ in range(J * M // 2):  # mid-episode
        src.random_step(seed=1)
    return src, envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)


def time_gather(B, J, M, E, flush):
    src, dst = env_pair(B, J, M, E)
    idx = torch.randperm(B, device="cuda").to(torch.int32)
    lib = src._lib
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda: lib.mtfjsp_gather(dst._h, src._h, C.c_void_p(idx.data_ptr()), stream)
    per_env = int(lib.mtfjsp_bytes_per_gather(dst._h))

    def med(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(20):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    assert call() == 0
    us = med(call)
    us_py = med(lambda: dst.gather_from(src, idx))
    return {"envs": B, "size": "J%dM%dE%d" % (J, M, E), "bytes_per_env": per_env, "gather_kernel_us": us,
            "gather_GB_per_s": B * per_env / (us * 1e-6) / 1e9, "gather_from_us": us_py}


def _labelled(owner, name, label):
    f = getattr(owner, name)

    def g(*a, **k):
        with torch.profiler.record_function(label):
            return f(*a, **k)

    setattr(owner, name, g)


def breakdown(job, mch, inst, W):
    """(c): per-stage host time and per-kernel device time of one beam_validate call, per step (36 steps)."""
    N = inst["t"].shape[1]
    for owner, name, label in ((job, "evaluate", "stage: job actor"), (mch, "forward", "stage: machine actor"),
                               (envm.BatchedMTFJSPEnv, "mfea1", "stage: candidate-machine features (mfea1)"),
                               (envm.BatchedMTFJSPEnv, "gather_from", "stage: gather_from"),
                               (envm.BatchedMTFJSPEnv, "step_obs", "stage: env step_obs"),
                               (val, "beam_select", "stage: selection (sort)")):
        _labelled(owner, name, label)
    val.beam_validate(job, mch, inst, W)
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        t, _ = wall(lambda: val.beam_validate(job, mch, inst, W))
    ev = prof.key_averages()
    dev = lambda e: float(getattr(e, "self_device_time_total", getattr(e, "self_cuda_time_total", 0.0)))
    # a host range appears twice (its host side and its span on the device timeline): the host side has the CPU time
    stage = [e for e in ev if e.key.startswith("stage: ") and e.cpu_time_total > 0]
    kernels = sorted(((e.key, dev(e) / N / 1e3, e.count / N) for e in ev
                      if dev(e) > 0 and not e.key.startswith("stage: ") and "CUDA" in str(getattr(e, "device_type", ""))),
                     key=lambda x: -x[1])
    return {"W": W, "profiled_total_s": t, "profiled_ms_per_step": t / N * 1e3,
            "host_ms_per_step_by_stage": {e.key[7:]: e.cpu_time_total / N / 1e3 for e in stage},
            "device_ms_per_step_all_kernels_and_copies": sum(k[1] for k in kernels),
            "device_ops_per_step": sum(k[2] for k in kernels),
            "top_kernels_ms_per_step": [{"name": k[0][:120], "ms": k[1], "launches": k[2]} for k in kernels[:15]],
            "table": ev.table(sort_by="self_cpu_time_total", row_limit=30)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "beam_b200.json")
    res = {"gpu": gpu_info()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res["gather"] = [time_gather(B, J, M, E, flush) for B, J, M, E in ((4096, 6, 6, 2), (65536, 6, 6, 2), (4096, 30, 20, 5))]
    del flush
    print(json.dumps(res["gather"], indent=1), flush=True)

    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    S, N = inst["t"].shape[:2]
    res["beam"] = []
    for tag in ("iotj", "n12800"):
        sd_op, sd_m = val.load_actor_state_dicts(g, tag)
        for prec in ("tf32", "fp32"):
            job, mch = enc.JobActor(sd_op, 6, 6, precision=prec), enc.MachineActor(sd_m, 6, precision=prec)
            greedy = val.greedy_validate(job, mch, inst, chunk=S)["objective"]
            row = {"checkpoint": tag, "precision": prec, "greedy_mean_objective": float(greedy.mean()), "widths": []}
            for W in WIDTHS:
                val.beam_validate(job, mch, inst, W)  # warm-up of this W's shapes
                runs = [wall(lambda: val.beam_validate(job, mch, inst, W)) for _ in range(3)]
                t, out = float(np.median([r[0] for r in runs])), runs[0][1]
                smp = val.sampled_validate(job, mch, inst, samples=W, seed=0)
                row["widths"].append({"W": W, "total_s": t, "total_s_runs": [r[0] for r in runs], "per_step_ms": t / N * 1e3,
                                      "beam_mean_best_objective": float(out["best_objective"].mean()),
                                      "live_slots_at_end": int(out["alive"].sum()),
                                      "instances_beam_better_than_greedy": int((out["best_objective"] < greedy - 1e-12).sum()),
                                      "instances_beam_worse_than_greedy": int((out["best_objective"] > greedy + 1e-12).sum()),
                                      "sampled_K_eq_W_mean_best_objective": float(smp["best_objective"].mean())})
                print(json.dumps({"checkpoint": tag, "precision": prec, **row["widths"][-1]}), flush=True)
            res["beam"].append(row)
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    res["breakdown"] = breakdown(enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32"), inst, 4)
    print(json.dumps(res["breakdown"], indent=1), flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(txt)


if __name__ == "__main__":
    main()
