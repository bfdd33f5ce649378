"""Host-buffer step (mtfjsp_step_host_packed, bench.py's e2e) and its parts alone: the packed H2D copy, the fused kernel
over the whole batch, the packed D2H copy, an empty graph launch + synchronize.    python profiles/prof_host_step.py [A|B|C]"""
import importlib
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402

wl = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "A"]
pkg = importlib.import_module("e2e-mappo-for-mt-fjsp_b200")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
J, M, E, B = wl["J"], wl["M"], wl["E"], wl["B"]
N = J * M
d = pkg.instances.synthetic_instances(0, B, J, M, E, wl["seed"])
w = pkg.instances.random_weights(0, B, wl["seed"])


env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
env.load(d["t"], d["p"], d["transT"], d["edge"])
env.scaler_init()
env.reset(w)
rec_op = torch.empty((N, B), dtype=torch.int32, device="cuda")
rec_mc = torch.empty((N, B), dtype=torch.int32, device="cuda")
for s in range(N):
    env.random_step(seed=99)
    rec_op[s].copy_(env.op); rec_mc[s].copy_(env.mach)
h_act = torch.stack([rec_op.cpu(), rec_mc.cpu()], dim=2).contiguous().pin_memory()
act_ptr = [h_act[s].data_ptr() for s in range(N)]

_, h_rec = env.host_buffers()
step = env.host_stepper(h_rec)
best = 1e9
for rep in range(4):
    env.reset(w); env.scaler_reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(N):
        step(act_ptr[s])
    torch.cuda.synchronize()
    best = min(best, (time.perf_counter() - t0) / N)
print("host step: %.1f us per %d-env step -> %.3e env-steps/s" % (best * 1e6, B, B / best), flush=True)

# the parts alone
nbytes = int(env._lib.mtfjsp_host_record_bytes(env._h))
dev_rec = torch.empty((B, nbytes), dtype=torch.uint8, device="cuda")
host_rec = torch.empty((B, nbytes), dtype=torch.uint8).pin_memory()
dev_act = torch.empty((B, 2), dtype=torch.int32, device="cuda")


def timeit(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e6


print("H2D %d B: %.1f us; D2H %d B: %.1f us" % (B * 8, timeit(lambda: dev_act.copy_(h_act[0], non_blocking=True)), B * nbytes,
                                                timeit(lambda: host_rec.copy_(dev_rec, non_blocking=True))))
env.reset(w); env.scaler_reset()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
tot = 0.0
for s in range(N):
    ev[0].record(); env.step_obs(rec_op[s], rec_mc[s]); ev[1].record(); torch.cuda.synchronize(); tot += ev[0].elapsed_time(ev[1])
print("fused step+obs kernel over the whole batch: %.1f us" % (tot / N * 1e3))
g = torch.cuda.CUDAGraph()
x = torch.zeros(1, device="cuda")
with torch.cuda.graph(g):
    x.add_(1)


def launch_sync():
    g.replay(); torch.cuda.synchronize()


t0 = time.perf_counter()
for _ in range(200):
    launch_sync()
print("one-node graph launch + synchronize: %.1f us" % ((time.perf_counter() - t0) / 200 * 1e6))
