"""Times the UNMODIFIED Python reference on this host (SURVEY.md 8(d) i): trainer/parallel_env.Parallel_env over
networkx, batch 16, J6M6E2 instances of the reference generator's seed-0 stream, random valid actions under the ESA
job mask, each step = cal_cur_task_machine_feature + DGFJSPEnv_paral_step + job-mask update, one process = one core.

TEST / BASELINE INFRASTRUCTURE ONLY (bench.py's cpu_baseline_reference leg runs it in a subprocess).  The reference tree
is read from $MTFJSP_REFERENCE_ROOT.

    python oracle/time_reference.py --seconds 12 --seed 0   ->  {"env_steps_per_s": ..., ...}
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=12.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--batch", type=int, default=16)
    a = ap.parse_args()
    import importlib.util

    from oracle import ref_harness as rh

    spec = importlib.util.spec_from_file_location("instances", os.path.join(os.path.dirname(HERE), "e2e-mappo-for-mt-fjsp_b200", "instances.py"))
    ins = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ins)
    import torch

    torch.set_num_threads(1)
    J, M, E, B = 6, 6, 2, a.batch
    N = J * M
    ref = rh.load_reference()
    d = ins.reference_stream_instances(B * (a.seed + 1), J, M, E, seed=0)  # the training stream; process p takes its own 16
    sl = slice(B * a.seed, B * (a.seed + 1))
    t, p, tt, edge = d["t"][sl], d["p"][sl], d["transT"][sl], d["edge"][sl]
    rng = np.random.default_rng(a.seed)
    args = rh.make_args(J, M, E, B)
    steps, t_run = 0, 0.0
    first = True
    while True:
        with contextlib.redirect_stdout(io.StringIO()):
            pe = ref.Parallel_env(args)
            pe.ability_instance = [[t[b].copy(), p[b].copy(), tt[b].copy(), np.array(edge[b])] for b in range(B)]
            pe.init_RewardScaling_sameBATCH(shape=4)
            adj, mfea2, tfea = pe.init_DGFJSPEnv_state0()      # unmodified constructor + reset path (parallel_env.py:87-142)
            jm = rh.RealJobMask(J, M, B)
            cand, mask = jm.initial()
            t0 = time.perf_counter()
            for s in range(N):
                jobs = np.array([rng.choice(np.nonzero(~mask[b])[0]) for b in range(B)])
                ops = cand[np.arange(B), jobs]
                mch = np.array([rng.choice(np.nonzero(t[b, ops[b]] >= 0)[0]) for b in range(B)])
                mmask = torch.tensor(np.stack([~(t[b, ops[b]] >= 0) for b in range(B)])[:, None, :])
                pe.cal_cur_task_machine_feature(torch.tensor(ops), mmask, tfea)
                adj, info, mfea2, tfea = pe.DGFJSPEnv_paral_step(list(zip(ops.tolist(), mch.tolist())))
                cand, mask = jm.update(pe, jobs)
            dt = time.perf_counter() - t0
        if first:
            first = False          # warm-up episode (imports, allocator)
            continue
        steps += N * B
        t_run += dt
        if t_run >= a.seconds:
            break
    print(json.dumps({"env_steps_per_s": steps / t_run, "env_steps": steps, "seconds": t_run, "batch": B, "seed": a.seed}))


if __name__ == "__main__":
    main()
