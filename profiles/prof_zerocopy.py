"""Host-buffer packed step (mtfjsp_step_host_packed, bench.py's e2e) with pinned buffers, by MTFJSP_HOST_ZEROCOPY level:
1 = one launch whose warps write the records straight into the mapped pinned host buffer, the actions copied in first,
2 = the actions are read from mapped host memory in place too.  The checksum of the last records lets two builds of the
library (MTFJSP_LIB) be compared on the same inputs.
    python profiles/prof_zerocopy.py [A|B|C]     a bench.WORKLOADS key
    python profiles/prof_zerocopy.py J M E B     any size (synthetic instances, seed 0)"""
import hashlib
import importlib
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402

if len(sys.argv) == 5:
    J, M, E, B = (int(x) for x in sys.argv[1:])
    seed = 0
else:
    wl = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "A"]
    J, M, E, B, seed = wl["J"], wl["M"], wl["E"], wl["B"], wl["seed"]
pkg = importlib.import_module("e2e-mappo-for-mt-fjsp_b200")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
N = J * M
d = pkg.instances.synthetic_instances(0, B, J, M, E, seed)
w = pkg.instances.random_weights(0, B, seed)


def make(level):
    os.environ["MTFJSP_HOST_ZEROCOPY"] = str(level)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    return env


env = make(1)
rec_op = torch.empty((N, B), dtype=torch.int32, device="cuda")
rec_mc = torch.empty((N, B), dtype=torch.int32, device="cuda")
for s in range(N):
    env.random_step(seed=99)
    rec_op[s].copy_(env.op); rec_mc[s].copy_(env.mach)
h_act = torch.stack([rec_op.cpu(), rec_mc.cpu()], dim=2).contiguous().pin_memory()
act_ptr = [h_act[s].data_ptr() for s in range(N)]

print("J%dM%dE%d x %d envs, %s" % (J, M, E, B, torch.cuda.get_device_name()), flush=True)
ref = None
for level in (1, 2, 2, 1):
    env = make(level)
    _, h_rec = env.host_buffers()
    step = env.host_stepper(h_rec)
    ts = []
    for rep in range(6):
        env.reset(w); env.scaler_reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(N):
            step(act_ptr[s])
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) / N)
    ts.sort()
    med = 0.5 * (ts[2] + ts[3])
    final = h_rec.clone()
    if ref is None:
        ref = final
    same = bool(torch.equal(final, ref))
    print("zerocopy %d: median %.1f us (min %.1f) per %d-env step -> %.3e env-steps/s; last records identical to level 1: "
          "%s, sha1 %s" % (level, med * 1e6, ts[0] * 1e6, B, B / med, same, hashlib.sha1(final.numpy().tobytes()).hexdigest()[:16]),
          flush=True)
