"""Knob experiments for the env kernel and the host-buffer step (one process per setting; the knobs are read from
the environment when the handle is created; MTFJSP_HOST_ZEROCOPY=2 reads the host step's actions in place, 1 copies them):

    MTFJSP_HOST_ZEROCOPY=1|2  MTFJSP_FUSE_POLICY=0|1  MTFJSP_OBS_INCREMENTAL=0|1  python profiles/exp_knobs.py [workload] [reps]

Prints one JSON line: fused-kernel time per launch (CUDA events around each launch, recorded actions replayed),
whole random-rollout step time, and the host-buffer step rate."""
import importlib
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402

wl = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "A"]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
pkg = importlib.import_module("e2e-mappo-for-mt-fjsp_b200")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
J, M, E, B = wl["J"], wl["M"], wl["E"], wl["B"]
N = J * M
d = pkg.instances.synthetic_instances(0, B, J, M, E, wl["seed"])
w = torch.as_tensor(pkg.instances.random_weights(0, B, wl["seed"])).cuda()
env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
env.load(d["t"], d["p"], d["transT"], d["edge"])
env.scaler_init()
env.reset(w)
rec_op = torch.empty((N, B), dtype=torch.int32, device="cuda")
rec_mc = torch.empty((N, B), dtype=torch.int32, device="cuda")
for s in range(N):
    env.random_step(seed=99)
    rec_op[s].copy_(env.op); rec_mc[s].copy_(env.mach)
assert int(env.done.sum()) == B and int(env.invalid.sum()) == 0
costs_ref = env.costs().clone()

evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(N)]
kms = 0.0
for rep in range(reps + 1):
    env.reset(w); env.scaler_reset()
    for s in range(N):
        evs[s][0].record(); env.step_obs(rec_op[s], rec_mc[s]); evs[s][1].record()
    torch.cuda.synchronize()
    if rep:
        kms += sum(a.elapsed_time(b) for a, b in evs)
k_us = kms * 1e3 / (reps * N)
assert torch.equal(env.costs(), costs_ref)

# whole random-rollout step (policy + mfea1 + fused kernel)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
env.reset(w); env.scaler_reset()
e0.record()
for rep in range(reps):
    for s in range(N):
        env.random_step(seed=5 + rep)
    env.reset(w); env.scaler_reset()
e1.record(); torch.cuda.synchronize()
r_us = e0.elapsed_time(e1) * 1e3 / (reps * N)

# host-buffer step
h_op = rec_op.cpu().pin_memory(); h_mc = rec_mc.cpu().pin_memory()
info6 = torch.empty((B, 6), dtype=torch.float64).pin_memory()
h_jm = torch.empty((B, J), dtype=torch.uint8).pin_memory()
h_cd = torch.empty((B, J), dtype=torch.int32).pin_memory()


def host_episode():
    env.reset(w); env.scaler_reset()
    for s in range(N):
        env.step_host(h_op[s], h_mc[s], info6, h_jm, h_cd)


host_episode()
torch.cuda.synchronize()
t0 = time.perf_counter()
for rep in range(reps):
    host_episode()
torch.cuda.synchronize()
h_us = (time.perf_counter() - t0) * 1e6 / (reps * N)
assert float(info6[:, 1].sum()) == B and torch.equal(env.costs(), costs_ref)

# packed host-buffer step
p_act, p_rec = env.host_buffers()
p_acts = torch.stack([rec_op.cpu(), rec_mc.cpu()], dim=2).contiguous().pin_memory()  # [N,B,2]


def packed_episode():
    env.reset(w); env.scaler_reset()
    for s in range(N):
        env.step_host_packed(p_acts[s], p_rec)


packed_episode()
torch.cuda.synchronize()
t0 = time.perf_counter()
for rep in range(reps):
    packed_episode()
torch.cuda.synchronize()
p_us = (time.perf_counter() - t0) * 1e6 / (reps * N)
recv = p_rec.numpy().view(env.host_record_dtype())[:, 0]
assert float(recv["done"].sum()) == B and torch.equal(env.costs(), costs_ref)
bytes_step = env.bytes_per_step()
print(json.dumps({"workload": sys.argv[1] if len(sys.argv) > 1 else "A",
                  "knobs": {k: v for k, v in os.environ.items() if k.startswith("MTFJSP_")},
                  "kernel_us": round(k_us, 2), "hbm_frac": round(bytes_step * B / (k_us * 1e-6) / 1e9 / bench.measured_peak()[0], 4),
                  "rollout_step_us": round(r_us, 2), "host_step_us": round(h_us, 2), "host_steps_per_s": round(B / (h_us * 1e-6)),
                  "packed_step_us": round(p_us, 2), "packed_steps_per_s": round(B / (p_us * 1e-6))}))
