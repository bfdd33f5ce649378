"""ESA-PPO machine actor and ESA-driven rollouts at J6M6E2, 65,536 envs (profiles/README.md, "ESA-PPO baseline actors").

  forward   one machine-actor forward (scores, pooled, values) on the features of a live env batch, CUDA events around
            each call, the 126 MB L2 overwritten (256 MB memset) before every timed call; median of 60 calls:
              esa_fused   EsaMachineActor tf32 (stats + fold + head kernels, three small tcgen05 layers for pooled / bias)
              esa_layers  the same with MTFJSP_FUSED_ESA=0 (projections, BatchNorms, split first layer as separate launches)
              esa_fp32    EsaMachineActor fp32 (library FP32 GEMMs, the reference's arithmetic)
              mappo_tf32  MachineActor tf32 (GAT trunk in one launch + head in one launch), for comparison
  rollout   sampled rollouts under CUDA-graph replay (the configuration of bench.py's actor-driven rollout): env-steps/s
            over steps 5..36 of an episode, median of 5 episodes, ESA actors (both tf32) against the MAPPO actors.
  kernels   device time per kernel of the fused ESA forward (torch.profiler, separate from the timed calls).
Prints the results as JSON and also writes them to the path given as the first argument, if any."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")

B, J, M, E = 65536, 6, 6, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def time_calls(fn, n=60, warm=5):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)), "calls": n}


def make_env(seed=5):
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    w = ins.random_weights(0, B, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    return env, w


def forward_times():
    env, w = make_env()
    env.reset(w)
    env.obs(1)
    m1, mmask = env.mfea1(env.candidate[:, 0].contiguous())
    m2 = env.mach_fea
    h_o = torch.randn((B, 128), device="cuda")
    sd_esa = enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 22)
    sd_map = enc.seeded_state_dict(enc.machine_actor_keys(128), 12)
    out = {}
    with torch.no_grad():
        for name, mk, fused in (("esa_fused", lambda: enc.EsaMachineActor(sd_esa, M, precision="tf32"), True),
                                ("esa_layers", lambda: enc.EsaMachineActor(sd_esa, M, precision="tf32"), False),
                                ("esa_fp32", lambda: enc.EsaMachineActor(sd_esa, M, precision="fp32"), True),
                                ("mappo_tf32", lambda: enc.MachineActor(sd_map, M, precision="tf32"), True)):
            enc._FUSED_ESA = fused
            a = mk()
            out[name] = time_calls(lambda: a.forward(m1, m2, h_o, mmask, return_logits=True))
            print(name, out[name], flush=True)
        enc._FUSED_ESA = True
        ref = enc.EsaMachineActor(sd_esa, M, precision="fp32").forward(m1, m2, h_o, mmask, return_logits=True)[0]
        for fused in (True, False):
            enc._FUSED_ESA = fused
            s = enc.EsaMachineActor(sd_esa, M, precision="tf32").forward(m1, m2, h_o, mmask, return_logits=True)[0]
            out["max_abs_dev_scores_vs_fp32_" + ("fused" if fused else "layers")] = float((s - ref).abs().max())
        enc._FUSED_ESA = True
    out["scores_abs_max_fp32"] = float(ref.abs().max())
    out["fused_kernels_us_per_call"] = kernel_breakdown(lambda: enc.EsaMachineActor(sd_esa, M, precision="tf32"), (m1, m2, h_o, mmask))
    return out


def kernel_breakdown(mk, args, n=20):
    """Device time per kernel of one fused forward (torch.profiler, a run of its own after the timed ones)."""
    from torch.profiler import ProfilerActivity, profile

    a = mk()
    with torch.no_grad():
        for _ in range(3):
            a.forward(*args, return_logits=True)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                a.forward(*args, return_logits=True)
            torch.cuda.synchronize()
    rows = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if t > 0 and ev.count >= n:
            rows[ev.key[:90]] = round(t / n, 2)
    return dict(sorted(rows.items(), key=lambda kv: -kv[1]))


def rollout_rates():
    env, w = make_env(7)
    pairs = {
        "esa": (enc.EsaJobActor(enc.seeded_state_dict(enc.esa_job_actor_keys(128), 21), J, M, precision="tf32"),
                enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 22), M, precision="tf32")),
        "mappo": (enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M, precision="tf32"),
                  enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, precision="tf32")),
    }
    res = {}
    for rep in range(5):
        for name in ("mappo", "esa") if rep % 2 else ("esa", "mappo"):  # alternate the order
            job, mch = pairs[name]
            ro = rom.Rollout(env, job, mch, greedy=False, use_cuda_graph=True, seed=rep)
            ro.begin_episode(w)
            for _ in range(4):
                ro.step()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(env.N - 4):
                ro.step()
            b.record()
            b.synchronize()
            assert int(env.done.sum().item()) == B and int(env.invalid.sum().item()) == 0
            res.setdefault(name, []).append(B * (env.N - 4) / (a.elapsed_time(b) * 1e-3))
    return {k: {"median_env_steps_per_s": float(np.median(v)), "all": v} for k, v in res.items()}


def main():
    res = {"gpu": gpu_info(), "B": B, "size": "J6M6E2"}
    res["forward"] = forward_times()
    res["rollout"] = rollout_rates()
    print(json.dumps(res, indent=1))
    if len(sys.argv) > 1:
        json.dump(res, open(sys.argv[1], "w"), indent=1)


if __name__ == "__main__":
    main()
