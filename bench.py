#!/usr/bin/env python
"""bench.py -- MT-FJSP env-steps/sec on B200 (BASELINE.json metric), one JSON line on stdout.

A "step" is one pass of the environment hot path over the whole env batch: random valid action ->
candidate-machine features -> transition + reward + reward scaling + observation + job mask, i.e.
everything the environment side of Run.py's rollout loop does per step (SURVEY.md 3.1 / 8a rows a1-a12),
one launch of the fused kernel for the sizes that have a specialised one.  Episodes wrap inside the timed
region: every N = J*M steps the batch is reset (two more launches), as the reference's loop does.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload A|B|C] [--repeats R]
                    [--dump-outputs DIR]

The K-step timed region (barrier + synchronize on both sides, CUDA events, max over ranks) is repeated R >= 15 times
and the MEDIAN is reported, so that short runs (--steps 20 is a 1.8 ms region) are stable to < 2 %.  At N = 1 the same
invocation also measures BASELINE.json's configs[2] and configs[3] (`workloads`: J10M10E3 / 16,384 envs and J30M20E5 /
4,096 envs) and the transition kernel alone (`roofline.step_only`, north_star's ">= 50 % on the step kernel").

N > 1 is launched by the driver with torch.distributed.run; each rank owns its own env slice (weak
scaling, no data-path collective; NCCL is used only for the barrier and the max-over-ranks time).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1..3]
    "A": dict(name="J6M6E2 synthetic, 65536 envs/GPU, random-action rollouts", J=6, M=6, E=2, B=65536, seed=1002),
    "B": dict(name="J10M10E3 synthetic, 16384 envs/GPU, env step + mask/feature build", J=10, M=10, E=3, B=16384, seed=1003),
    "C": dict(name="J30M20E5 synthetic, 4096 envs/GPU", J=30, M=20, E=5, B=4096, seed=1004),
}
METRIC = "MT-FJSP env-steps/sec"
UNIT = "env-steps/s"


def workload_config(wl, B, world):
    """The `config` object of both arms (ours and --impl reference): it names the workload only, so the driver's
    same-config check compares like with like."""
    J, M, E = wl["J"], wl["M"], wl["E"]
    N = J * M
    survey = 8 + 2 * (18 * N + 42 * M + 8 * J + (N + 7) // 8 + 160) + (48 * N + 18 * N + 32 * M + 5 * J + 41)
    return {"workload": wl["name"], "envs_per_gpu": B, "jobs": J, "machines": M, "edges": E, "obs_dtype": "f32",
            "mask_mode": "ESA", "left_shift": True, "n_gpus": world,
            "l2": "working set %.0f MB per GPU > 126 MB L2 (inputs larger than L2)" % (B * (survey + 2000) / 1e6)}


def needed_bytes(J, M, fe, policy, rows_t, rows_a, rows_m):
    """Bytes ONE env-step of the incremental algorithm has to move (DESIGN.md "Roofline accounting"): the whole state is
    read (the reward needs the makespan and energy estimates over all ops), only what the step changes is written.
    State sizes are SURVEY.md 8(d)'s minimal array form, not this implementation's (fatter) records.
      read    B_state = 18N + 42M + 8J + ceil(N/8) + 160; the action (8) and t, p at (op, machine) (16) -- or, when the
              kernel draws the random action itself: job mask J + candidates 4J + step counter 2 + the op's t / p rows 16M
              + edge ids M
      write   changed state words 206 (op: machine, start, finish, link + successor's link 19; route count 2; scheduled
              bit 1; job's last finish 8; 4 scalars 32; one machine's accumulators 40; reward scaler 104)
              + 5 rewards, done 41 + 4 scaled rewards 32 + job mask and candidates 5J
              + changed observation rows (measured by diffing consecutive observations over one episode):
                rows_t x 12 fe + rows_a x 10 (ELL adjacency) + rows_m x 8 fe
              + with the in-kernel policy: the action 8, candidate-machine features 6 fe M, machine mask M"""
    N = J * M
    b_state = 18 * N + 42 * M + 8 * J + (N + 7) // 8 + 160
    rd = b_state + ((5 * J + 2 + 17 * M) if policy else 24)
    wr = 206 + 41 + 32 + 5 * J + rows_t * 12 * fe + rows_a * 10 + rows_m * 8 * fe
    if policy:
        wr += 8 + 6 * fe * M + M
    return {"total": rd + wr, "read": rd, "write": wr, "b_state": b_state,
            "changed_rows_per_step": {"task_fea": rows_t, "adjacency": rows_a, "mach_fea": rows_m}}


def median(xs):
    xs = sorted(xs)
    n = len(xs)
    return xs[n // 2] if n % 2 else 0.5 * (xs[n // 2 - 1] + xs[n // 2])


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_rate(wl, nthreads, target_seconds):
    """Times the CPU restatement (oracle/) on a bounded sample of the same workload: whole random rollouts,
    every step = mask + candidates + mfea1 + transition + reward + scaling + observation (oracle_rollout_random)."""
    from oracle.mtfjsp_oracle import OracleEnv

    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    J, M, E = wl["J"], wl["M"], wl["E"]
    N = J * M
    probe_B = max(nthreads * 4, 64 if N <= 100 else 16)

    def run(B, episodes):
        d = ins.synthetic_instances(0, B, J, M, E, wl["seed"])
        w = ins.random_weights(0, B, wl["seed"])
        o = OracleEnv(B, J, M, E, left_shift=True, nthreads=nthreads)
        o.load(d["t"], d["p"], d["transT"], d["edge"])
        o.scaler_init()
        o.reset(w)
        o.rollout_random(N, seed=1)  # warm-up episode
        t0 = time.perf_counter()
        for ep in range(episodes):
            o.reset(w)
            o.scaler_reset()
            o.rollout_random(N, seed=2 + ep)
        return B * N * episodes / (time.perf_counter() - t0)

    rate = run(probe_B, 1)
    B = int(min(max(probe_B, rate * target_seconds / (N * 4)), 262144))
    B = max(nthreads, (B // nthreads) * nthreads)
    rate = run(B, 4)
    return rate, "%d envs x 4 episodes x %d steps (%s), %d thread(s)" % (B, N, wl["name"].split(",")[0], nthreads)


def real_reference_rate(seconds=12.0):
    """SURVEY.md 8(d) i-ii: the UNMODIFIED Python reference (trainer/parallel_env.Parallel_env over networkx, batch 16,
    J6M6E2 instances of the shipped generator's seed-0 stream, random valid actions under the ESA mask) timed on this
    box's host cores: one process = one core (how the reference runs), then one process per core.  Needs a checkout of the
    reference project named by $MTFJSP_REFERENCE_ROOT; the leg is left out without one."""
    ref_root = os.environ.get("MTFJSP_REFERENCE_ROOT", "")
    if not os.path.isdir(os.path.join(ref_root, "graph-jsp-env", "src", "graph_jsp_env")):
        return None
    script = os.path.join(ROOT, "oracle", "time_reference.py")
    env = dict(os.environ, MTFJSP_REFERENCE_ROOT=ref_root, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1

    def run(nproc):
        ps = [subprocess.Popen([sys.executable, script, "--seconds", str(seconds), "--seed", str(p)], env=env,
                               stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for p in range(nproc)]
        rates = []
        for pr in ps:
            out, _ = pr.communicate(timeout=seconds * 6 + 120)
            for ln in out.splitlines():
                if ln.startswith("{"):
                    rates.append(json.loads(ln)["env_steps_per_s"])
        return rates

    try:
        one = run(1)
        allc = run(cores)
    except Exception as e:  # a baseline leg must never take the bench line down
        return {"error": repr(e)[:200]}
    if not one or not allc:
        return {"error": "reference timing produced no output"}
    return {"value": one[0], "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": "unmodified trainer/parallel_env.Parallel_env, 16 envs J6M6E2 (generator seed 0), whole random "
                      "episodes for %.0f s incl. cal_cur_task_machine_feature + job-mask update" % seconds,
            "all_cores": {"value": sum(allc), "cores": cores, "processes": len(allc)}}


def run_reference(args, wl):
    """--impl reference: the reference's algorithm on the host cores.  The reference itself is Python over networkx
    (157 env-steps/s per core, BASELINE.md); this arm times its C restatement (oracle/, kind 'port') with all host
    threads on the SAME workload, batch and step definition as our arm: one step = one env-step of every env of the
    batch (random valid action + candidate-machine features + transition + reward + scaling + observation + mask)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.mtfjsp_oracle import OracleEnv

    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    # every host core this process may run on (torchrun exports OMP_NUM_THREADS=1; the oracle's parallel loops take an
    # explicit thread count, so that default does not starve the reference arm)
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    cores = max(1, cores)
    J, M, E, B = wl["J"], wl["M"], wl["E"], args.batch or wl["B"]
    N = J * M
    d = ins.synthetic_instances(0, B, J, M, E, wl["seed"])
    w = ins.random_weights(0, B, wl["seed"])
    o = OracleEnv(B, J, M, E, left_shift=True, nthreads=cores)
    o.load(d["t"], d["p"], d["transT"], d["edge"])
    o.scaler_init()
    o.reset(w)
    st = {"s": 0}

    def steps(n):
        while n > 0:
            if st["s"] == N:
                o.reset(w); o.scaler_reset(); st["s"] = 0
            k = min(n, N - st["s"])
            o.rollout_random(k, seed=1234)
            st["s"] += k
            n -= k

    K, W = args.steps, max(args.warmup, 3)
    t_all = time.perf_counter()
    steps(W)
    times = []
    # bounded: the whole arm ends within a few minutes whatever K is
    while len(times) < args.repeats and (len(times) < 3 or time.perf_counter() - t_all < 150.0):
        t0 = time.perf_counter()
        steps(K)
        times.append(time.perf_counter() - t0)
    sec = median(times)
    val = B * K / sec
    sample = "%d envs x %d steps per timed region, median of %d regions (%s), %d thread(s)" % (
        B, K, len(times), wl["name"].split(",")[0], cores)
    line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": sec * 1e3 / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference", "config": workload_config(wl, B, args.gpus),
            "note": "CPU restatement of the reference env (oracle/, OpenMP over envs); the Python reference itself runs "
                    "~157 env-steps/s/core (BASELINE.md; re-timed on this box in our arm's cpu_baseline_reference)",
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "repeats": len(times), "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


DUMP_MAX_ENVS = 4096
DUMP_MAX_BYTES = 48 << 20


def snapshot_outputs(env, torch):
    """What `random_step` hands its caller (action, candidate-machine features, rewards, flags, observation, job mask and
    candidates) for a fixed, seeded sample of the batch's envs, as host float32 / float64 arrays.  Integer outputs are
    widened to float64, which holds them exactly."""
    import numpy as np

    outs = {"op": env.op, "mach": env.mach, "mfea1": env.mfea1_buf, "mach_mask": env.mach_mask, "reward5": env.reward5,
            "scaled4": env.scaled4, "done": env.done, "invalid": env.invalid, "task_fea": env.task_fea,
            "mach_fea": env.mach_fea, "adj_w": env.adj_w, "adj_src": env.adj_src, "job_mask": env.job_mask,
            "candidate": env.candidate}
    per_env = sum(x[0].numel() * 8 for x in outs.values())
    n = max(1, min(env.B, DUMP_MAX_ENVS, DUMP_MAX_BYTES // per_env))
    idx = np.sort(np.random.default_rng(0).choice(env.B, size=n, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    dump = {"env_index": idx.astype(np.float64)}
    for name, x in outs.items():
        y = x.index_select(0, sel).cpu()
        dump[name] = y.numpy() if y.dtype in (torch.float32, torch.float64) else y.to(torch.float64).numpy()
    return dump


def measure_env(wl, B, K, W, repeats, rank, world, dev, barrier, sh, envm, torch, want_e2e, want_dump=False):
    """Everything measured on one workload: whole-job throughput of the timed region, the kernels alone (one CUDA-event
    pair per launch on the launching stream), changed observation rows, and (want_e2e) the host-buffer C-ABI call.
    want_dump: also keep a sample of what the last timed step computed (snapshot_outputs)."""
    J, M, E = wl["J"], wl["M"], wl["E"]
    N = J * M
    first, count, d, w = sh.make_shard(B * world, rank, world, J, M, E, wl["seed"])
    assert count == B and first == rank * B
    w = torch.as_tensor(w).to(dev)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    state = {"s": 0}

    def one_step(seed=1234):
        if state["s"] == N:  # episode finished for every env: next episode (Run.py:615-665)
            env.reset(w)
            env.scaler_reset()
            state["s"] = 0
        env.random_step(seed=seed, env_offset=first)
        state["s"] += 1

    for _ in range(max(W, 3)):
        one_step()
    times, launches = [], 0
    for _ in range(repeats):
        barrier()
        l0 = env.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            one_step()
        e1.record()
        barrier()
        times.append(sh.max_over_ranks(e0.elapsed_time(e1), dev))
        launches = env.launch_count - l0
    ms = median(times)
    out = {"env": env, "first": first, "w": w, "d": d, "ms": ms, "times": times, "launches": launches,
           "value": B * world * K / (ms * 1e-3)}
    if want_dump:
        out["dump"] = snapshot_outputs(env, torch)

    # ---- record one episode of actions; count the observation rows a step changes (diff of consecutive observations) ----
    env.reset(w); env.scaler_reset()
    env.obs()
    rec_op = torch.empty((N, B), dtype=torch.int32, device=dev)
    rec_mc = torch.empty((N, B), dtype=torch.int32, device=dev)
    prev = [x.clone() for x in (env.task_fea, env.adj_w, env.adj_src, env.mach_fea)]
    rows = [0.0, 0.0, 0.0]
    for s in range(N):
        env.random_step(seed=99, env_offset=first)
        rec_op[s].copy_(env.op); rec_mc[s].copy_(env.mach)
        cur = (env.task_fea, env.adj_w, env.adj_src, env.mach_fea)
        rows[0] += float((cur[0] != prev[0]).any(-1).sum())
        rows[1] += float(((cur[1] != prev[1]).any(-1) | (cur[2] != prev[2])).sum())
        rows[2] += float((cur[3] != prev[3]).any(-1).sum())
        for a, b in zip(prev, cur):
            a.copy_(b)
    del prev
    assert int(env.done.sum().item()) == B and int(env.invalid.sum().item()) == 0
    rows = [r / (N * B) for r in rows]
    out["rec_op"], out["rec_mc"] = rec_op, rec_mc

    # ---- kernels alone ----
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(N)]
    reps = max(2, min(6, (4 * 36) // N + 1))

    def per_launch_us(launch):
        tot, n = 0.0, 0
        for rep in range(reps + 1):
            env.reset(w); env.scaler_reset()
            for s in range(N):
                evs[s][0].record()
                launch(s, rep)
                evs[s][1].record()
            torch.cuda.synchronize()
            if rep > 0:  # first replay is warm-up
                tot += sum(a.elapsed_time(b) for a, b in evs)
                n += N
        return tot * 1e3 / n

    peak, peak_src = measured_peak()
    gbs = lambda nbytes, us: nbytes * B / (us * 1e-6) / 1e9
    b_state = 18 * N + 42 * M + 8 * J + (N + 7) // 8 + 160
    kern = {}
    us = per_launch_us(lambda s, rep: env.step_obs(rec_op[s], rec_mc[s]))
    nb, sb = needed_bytes(J, M, 4, False, *rows), env.bytes_per_step()
    kern["step_obs"] = {"kernel": "env_kernel_s<STEP|OBS,float> (actions given: the actor-driven and host-step paths)",
                        "kernel_us": us, "bytes_per_env_step": nb["total"], "achieved": gbs(nb["total"], us),
                        "frac": gbs(nb["total"], us) / peak, "bytes_survey_full_rewrite": sb,
                        "frac_survey_bytes": gbs(sb, us) / peak}
    us = per_launch_us(lambda s, rep: env.step(rec_op[s], rec_mc[s]))
    so = 8 + 2 * b_state + 41
    kern["step_only"] = {"kernel": "env_kernel_s<STEP,double> (mtfjsp_step: transition + reward + reward scaling + job mask, "
                                   "no observation)", "kernel_us": us, "bytes_per_env_step": so,
                         "bytes_accounting": "SURVEY.md 8(d): 8 + 2*B_state + 41", "achieved": gbs(so, us),
                         "frac": gbs(so, us) / peak, "steps_per_s_kernel_only": B / (us * 1e-6)}
    if env.random_step_is_fused:
        us = per_launch_us(lambda s, rep: env.random_step(seed=500 + rep, env_offset=first))
        nb, sb = needed_bytes(J, M, 4, True, *rows), env.bytes_per_random_step()
        kern["random_step"] = {"kernel": "env_kernel_s<STEP|OBS|POLICY,float> (random policy + candidate-machine features + "
                                         "step + reward + observation + job mask; the kernel of the timed region)",
                               "kernel_us": us, "bytes_per_env_step": nb["total"], "achieved": gbs(nb["total"], us),
                               "frac": gbs(nb["total"], us) / peak, "bytes_terms": nb, "bytes_survey_full_rewrite": sb,
                               "frac_survey_bytes": gbs(sb, us) / peak, "steps_per_s_kernel_only": B / (us * 1e-6)}
    out["kern"], out["peak"], out["peak_src"], out["rows"] = kern, peak, peak_src, rows

    # ---- e2e: host-buffer C-ABI call per step (pinned H2D action pairs, D2H packed step records = step info + job
    # mask + candidates; mtfjsp_step_host_packed: one launch whose warps write their records straight into the mapped pinned
    # host buffer and read the action pairs from it -- the bytes below cross PCIe inside the timed region, by SM loads /
    # stores instead of the copy engine) ----
    if want_e2e:
        h_act = torch.stack([rec_op.cpu(), rec_mc.cpu()], dim=2).contiguous().pin_memory()  # [N,B,2] (op, machine)
        _, h_rec = env.host_buffers()
        rec_view = h_rec.numpy().view(env.host_record_dtype())[:, 0]
        host_step = env.host_stepper(h_rec)                       # prepared call: buffers bound once
        act_ptr = [h_act[s].data_ptr() for s in range(N)]         # this step's pinned [B,2] action array
        es = {"s": N}

        def e2e_steps(n):
            for _ in range(n):
                if es["s"] == N:
                    env.reset(w); env.scaler_reset(); es["s"] = 0
                host_step(act_ptr[es["s"]])
                es["s"] += 1

        e2e_steps(N + 3)  # one whole episode first: every action buffer's graph is instantiated outside the timed region
        Ke = min(K, 4 * N)
        et = []
        for _ in range(repeats):
            barrier()
            t0 = time.perf_counter()
            e2e_steps(Ke)
            torch.cuda.synchronize()
            et.append(sh.max_over_ranks(time.perf_counter() - t0, dev))
        e2e_s = median(et)
        out["e2e"] = {"value": B * world * Ke / e2e_s, "unit": UNIT, "h2d_bytes_per_step": B * 8,
                      "d2h_bytes_per_step": B * h_rec.shape[1],
                      "api": "mtfjsp_step_host_packed (C ABI, pinned host buffers: [B,2] i32 action pairs in, [B] packed "
                             "records (f64 r, f64 scaled[4], u8 done, job-mask bits, u8 next op per job) out, written by the step kernel itself over "
                             "PCIe (mapped host memory); observation tensors stay on the device)",
                      "steps": Ke, "repeats": repeats, "us_per_step": e2e_s * 1e6 / Ke}
        assert float(rec_view["done"].sum()) in (0.0, float(B))
        # the same call returning ONLY the reference's step info (`oenv_info` rows, 48 B per env): candidates and job mask
        # stay on the device, where the actors that consume them run (mtfjsp_step_host with NULL mask / candidate buffers)
        h_op = [rec_op[s].cpu().pin_memory() for s in range(N)]
        h_mc = [rec_mc[s].cpu().pin_memory() for s in range(N)]
        h_info = torch.zeros((B, 6), dtype=torch.float64).pin_memory()

        def info_steps(n):
            for _ in range(n):
                if es["s"] == N:
                    env.reset(w); env.scaler_reset(); es["s"] = 0
                env.step_host(h_op[es["s"]], h_mc[es["s"]], h_info, None, None)
                es["s"] += 1

        es["s"] = N
        info_steps(N + 3)
        it = []
        for _ in range(max(3, repeats // 3)):
            barrier()
            t0 = time.perf_counter()
            info_steps(Ke)
            torch.cuda.synchronize()
            it.append(sh.max_over_ranks(time.perf_counter() - t0, dev))
        out["e2e"]["step_info_only"] = {"value": B * world * Ke / median(it), "unit": UNIT, "h2d_bytes_per_step": B * 8,
                                        "d2h_bytes_per_step": B * 48, "us_per_step": median(it) * 1e6 / Ke,
                                        "api": "mtfjsp_step_host (op / machine arrays in, the [B,6] float64 step info of "
                                               "trainer/parallel_env.py:260 out; candidates, job mask and observation stay "
                                               "on the device)"}
    return out


def kernel_traffic(J, M, B):
    """ncu --set full DRAM bytes per launch of the env kernels on this workload (profiles/r02_env_kernel_traffic.json,
    written from this round's captures by profiles/ncu_traffic.py), or {}."""
    for name in ("r02_env_kernel_traffic.json",):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            try:
                return json.load(open(path)).get("J%dM%d_B%d" % (J, M, B), {})
            except Exception:
                pass
    return {}


def run_ours(args, wl):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stdout_fd = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries the one JSON line only: NCCL prints its version banner with printf when NCCL_DEBUG=VERSION, so
        # everything the libraries write to fd 1 goes to stderr until the line is printed
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    sh = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.sharding")
    J, M, E, B = wl["J"], wl["M"], wl["E"], args.batch or wl["B"]
    if args.scaling == "strong":  # fixed total batch: the workload's env count is split over the ranks
        B = max(1, B // world)
    N = J * M
    K, W, R = args.steps, args.warmup, max(1, args.repeats)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # weak scaling: B envs per GPU, env i of the B*world job lives on rank i // B (contiguous slices)
    mm = measure_env(wl, B, K, W, R, rank, world, dev, barrier, sh, envm, torch, want_e2e=True,
                     want_dump=bool(args.dump_outputs) and rank == 0)
    env, first, w, d = mm["env"], mm["first"], mm["w"], mm["d"]
    rec_op, rec_mc = mm["rec_op"], mm["rec_mc"]
    ms, value, launches, peak, peak_src, kern = mm["ms"], mm["value"], mm["launches"], mm["peak"], mm["peak_src"], mm["kern"]
    h_op = rec_op.cpu(); h_mc = rec_mc.cpu()
    # ---- BASELINE.json configs[4] (forward half): the same env slice driven by the MAPPO actors on the device ----
    policy = None
    if not args.no_policy and (J, M) == (6, 6):
        enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
        rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
        job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M, precision="tf32")
        mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, precision="tf32")
        ro = rom.Rollout(env, job, mch, greedy=False, use_cuda_graph=True, seed=1)
        ro.begin_episode(w)
        for _ in range(4):
            ro.step()  # eager first step, warm-up, capture
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nstep = N - 4
        p0.record()
        for _ in range(nstep):
            ro.step()
        p1.record()
        barrier()
        pms = sh.max_over_ranks(p0.elapsed_time(p1), dev)
        assert int(env.done.sum().item()) == B and int(env.invalid.sum().item()) == 0
        policy = {"value": B * world * nstep / (pms * 1e-3), "unit": UNIT, "ms_per_step": pms / nstep, "steps": nstep,
                  "what": "job actor (GIN encoder: tcgen05 TF32 layers fed by TMA, aggregation in the layer's epilogue; policy head "
                          "in one launch) + machine actor (GAT trunk in one launch, head in one launch) + one-launch action "
                          "selection + env step/obs, CUDA-graph replay, random-init weights", "hidden": 128}
    stats = sh.reduce_episode_stats(env.costs(), device=dev)  # the rollout side's only other exchange (6 doubles)

    # ---- BASELINE.json configs[4]: env slice + encoder + PPO update end to end, gradient allreduce share ----
    train = None
    if not args.no_train and (J, M) == (6, 6):
        enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
        rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
        ppo = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.ppo")
        Bt = min(B, 8192)  # 65,536 envs over 8 GPUs
        env_t = envm.BatchedMTFJSPEnv(Bt, J, M, E, left_shift=True, obs_dtype=torch.float32)
        env_t.load(d["t"][:Bt], d["p"][:Bt], d["transT"][:Bt], d["edge"][:Bt])
        env_t.scaler_init()
        tj = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M, trainable=True)
        tm = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, trainable=True)
        tc = enc.GlobalCritic(enc.seeded_state_dict(enc.global_critic_keys(128), 13), J, M, trainable=True)
        tro = rom.Rollout(env_t, tj.inference_twin("tf32"), tm.inference_twin("tf32"), greedy=False, use_cuda_graph=True,
                          seed=2 + rank)
        wt = [w[:Bt]]
        runs = {}
        for variant, enc_tf32 in (("tcgen05_tf32", True), ("library_fp32", False)):
            up = ppo.MAPPOUpdate(tj, tm, tc, ppo.PPOConfig(k_epochs=1, encoder_tf32=enc_tf32))
            tms, cms, ams = [], [], []
            for it in range(4):  # first iteration is warm-up (library initialisation); median of the other three
                barrier()
                t0e, t1e, t2e = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                t0e.record()
                btc = ppo.collect(tro, wt)
                t1e.record()
                up.recompute_old_logp(btc)       # the TF32 twins collected it: behaviour log-probs on the update's path
                losses, _ = up.update(btc, N)    # (refreshes the twins' cached weight layouts at the end)
                t2e.record()
                barrier()
                a_ms = up.allreduce_ms()
                if it > 0:
                    cms.append(sh.max_over_ranks(t0e.elapsed_time(t1e), dev)); tms.append(sh.max_over_ranks(t0e.elapsed_time(t2e), dev))
                    ams.append(a_ms)
                buf_bytes = btc.bytes_per_env_step()
                del btc
            k_med = sorted(range(len(tms)), key=lambda i_: tms[i_])[len(tms) // 2]  # the iteration with the median total time
            runs[variant] = (tms[k_med], cms[k_med], ams[k_med], [float(x) for x in losses], up.allreduce_bytes // 4)
        tot, col, arm, losses, arb = runs["tcgen05_tf32"]
        train = {"value": Bt * world * N / (tot * 1e-3), "unit": UNIT, "envs_per_gpu": Bt, "buffer_steps": N, "k_epochs": 1,
                 "mini_bs": N, "collect_ms": col, "update_ms": tot - col,
                 "allreduce_ms": arm, "allreduce_share": arm / tot,
                 "allreduce_bytes_per_update": arb, "losses": losses, "buffer_bytes_per_env_step": buf_bytes,
                 "update_ms_library_fp32": runs["library_fp32"][0] - runs["library_fp32"][1],
                 "value_library_fp32": Bt * world * N / (runs["library_fp32"][0] * 1e-3),
                 "what": "one buffer (1 episode) collected with the tcgen05 rollout twins (CUDA-graph replay) + one batched PPO "
                         "update; every [rows,128] x [128,<=128] product of the update (graph encoders, GAT projections, policy "
                         "heads) runs forward / input-gradient / weight-gradient on the hand-written tcgen05 TF32 kernels "
                         "(PPOConfig.encoder_tf32); aggregation, grouped BatchNorm and GAE kernels hand-written; NCCL gradient "
                         "allreduce when n_gpus > 1.  *_library_fp32 = the same update with every GEMM on the FP32 library path "
                         "(the reference's arithmetic)"}
        del env_t, up, tro
        torch.cuda.empty_cache()

    # ---- BASELINE.json configs[2], configs[3] in the same invocation (N = 1): value + kernel roofline ----
    others = {}
    if world == 1 and not args.no_workloads and args.workload == "A" and not args.batch:
        for key in ("B", "C"):
            wl2 = WORKLOADS[key]
            N2 = wl2["J"] * wl2["M"]
            m2 = measure_env(wl2, wl2["B"], N2, 3, 5, rank, world, dev, barrier, sh, envm, torch, want_e2e=False)
            k2 = m2["kern"]
            tr2 = kernel_traffic(wl2["J"], wl2["M"], wl2["B"])
            head2 = k2.get("random_step", k2["step_obs"])
            others[key] = {"config": workload_config(wl2, wl2["B"], world), "value": m2["value"], "unit": UNIT,
                           "steps": N2, "repeats": 5, "ms_per_step": m2["ms"] / N2,
                           "what": "whole episodes (%d steps) of the one-launch random-rollout step, median of 5" % N2,
                           "roofline": dict(head2, peak=peak, unit="GB/s", bound="hbm",
                                            traffic=tr2.get("random_step" if "random_step" in k2 else "step_obs")),
                           "step_obs_kernel": k2["step_obs"], "step_only": k2["step_only"]}
            del m2
            torch.cuda.empty_cache()

    clocks = sampler.stop() if sampler else None
    tr = kernel_traffic(J, M, B)
    headk = "random_step" if "random_step" in kern else "step_obs"
    head = kern[headk]
    traffic = tr.get(headk)

    # ---- the strict drop-in call: Parallel_env.DGFJSPEnv_paral_step with the reference's argument / return types
    # (python list of action pairs in, numpy float64 dense adjacency [B,N,N] + features + python info list out) ----
    dropin = None
    if rank == 0 and world == 1 and not args.no_dropin:
        pem = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.parallel_env")
        Bd = min(B, 8192)
        pe = pem.Parallel_env({"n_job": J, "n_machine": M, "n_edge": E, "env_batch": Bd, "GAMMA": 0.99,
                               "reward_scaling": {"scaling_divisor": 1}, "weight_mk": 0.4, "weight_ec": 0.4, "weight_tt": 0.2})
        pe.get_batch({k2: torch.as_tensor(d[k1][:Bd]) for k1, k2 in (("t", "t"), ("p", "p"), ("transT", "transT"), ("edge", "edge"))})
        pe.init_RewardScaling_sameBATCH(shape=4)
        pe.init_DGFJSPEnv_state0(weights=w[:Bd].cpu().numpy())
        acts = [list(zip(h_op[s2][:Bd].tolist(), h_mc[s2][:Bd].tolist())) for s2 in range(6)]
        pe.DGFJSPEnv_paral_step(acts[0])
        t0 = time.perf_counter()
        for s2 in range(1, 6):
            pe.DGFJSPEnv_paral_step(acts[s2])
        dt = time.perf_counter() - t0
        dropin = {"value": Bd * 5 / dt, "unit": UNIT, "envs": Bd, "d2h_bytes_per_step": Bd * (N * N * 8 + N * 96 + M * 64 + 80),
                  "api": "Parallel_env.DGFJSPEnv_paral_step (reference types: python action list in, numpy f64 dense "
                         "adjacency + features + python info list out)"}
        del pe
        # the same call with compat="ell": adjacency as (adj_w, adj_src) device tensors, only the [B,6] step info crosses PCIe
        pe = pem.Parallel_env({"n_job": J, "n_machine": M, "n_edge": E, "env_batch": Bd, "GAMMA": 0.99,
                               "reward_scaling": {"scaling_divisor": 1}, "weight_mk": 0.4, "weight_ec": 0.4, "weight_tt": 0.2},
                              compat="ell")
        pe.get_batch({k2: torch.as_tensor(d[k1][:Bd]) for k1, k2 in (("t", "t"), ("p", "p"), ("transT", "transT"), ("edge", "edge"))})
        pe.init_RewardScaling_sameBATCH(shape=4)
        pe.init_DGFJSPEnv_state0(weights=w[:Bd].cpu().numpy())
        acts_np = [np.stack((h_op[s2][:Bd].numpy(), h_mc[s2][:Bd].numpy()), axis=1) for s2 in range(12)]
        pe.DGFJSPEnv_paral_step(acts_np[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s2 in range(1, 12):
            pe.DGFJSPEnv_paral_step(acts_np[s2])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dropin["compat_ell"] = {"value": Bd * 11 / dt, "unit": UNIT, "envs": Bd, "d2h_bytes_per_step": Bd * 48,
                                "api": "Parallel_env(compat='ell').DGFJSPEnv_paral_step ([B,2] int array in; (adj_w, adj_src), "
                                       "features as device tensors and the [B,6] float64 step info out)"}
        del pe

    cpu = cpu_ref = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r1, sample = cpu_port_rate(wl, 1, 8.0)
        cpu = {"value": r1, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}
        if (J, M) == (6, 6):
            cpu_ref = real_reference_rate()

    if rank == 0:
        spread = (max(mm["times"]) - min(mm["times"])) / ms if ms else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(W, 3),
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(wl, B, world),
            "repeats": R, "timing": "median of %d timed regions of %d steps each (CUDA events, barrier + synchronize on "
                                    "both sides, max over ranks); (max-min)/median = %.3f" % (R, K, spread or 0.0),
            "impl_notes": {"parallelism": "env-slices x%d (no data-path collective)" % world,
                           "launches_per_step": round(launches / K, 3),
                           "kernels": "env_kernel_s<STEP|OBS|POLICY> (random policy + candidate-machine features + step + "
                                      "reward + obs + mask in one launch; reset launches reset_copy_kernel + scaler_kernel "
                                      "every %d steps)" % N},
            "e2e": mm["e2e"],
            "gpu_launches": launches,
            "roofline": dict(head, bound="hbm", peak=peak, unit="GB/s", traffic=traffic, peak_source=peak_src,
                             bytes_accounting="frac = bytes the incremental algorithm needs per env-step (needed_bytes() in "
                                              "bench.py: whole state read once in SURVEY 8(d)'s minimal form, changed state and "
                                              "changed observation rows written) / kernel time / peak; frac_survey_bytes = SURVEY "
                                              "8(d)'s full observation rewrite every step (what the reference does; round 1's "
                                              "headline); frac_of_peak_moved = ncu DRAM bytes of one launch / kernel time / peak",
                             frac_of_peak_moved=(traffic / (head["kernel_us"] * 1e-6) / 1e9 / peak) if traffic else None,
                             step_obs_kernel=dict(kern["step_obs"], traffic=tr.get("step_obs")),
                             step_only=dict(kern["step_only"], traffic=tr.get("step_only"))),
            "clocks": clocks,
            "episode_stats": {k: float(v) for k, v in stats.items()},
        }
        if others:
            line["workloads"] = others
        if policy:
            line["policy_rollout"] = policy
        if train:
            line["train_iteration"] = train
        if dropin:
            line["e2e"]["dropin_parallel_env"] = dropin
        if cpu:
            line["cpu_baseline"] = cpu
        if cpu_ref:
            line["cpu_baseline_reference"] = cpu_ref
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in mm["dump"].items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        if stdout_fd is not None:
            sys.stdout.flush()
            os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
        if stdout_fd is not None:
            os.dup2(2, 1)  # teardown chatter stays off stdout as well
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=360)
    ap.add_argument("--warmup", type=int, default=36)
    ap.add_argument("--repeats", type=int, default=15, help="timed regions of --steps steps each; the median is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="A", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, what the driver measures): the workload's env count per GPU; strong: that count in total")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-policy", action="store_true", help="skip the actor-driven rollout measurement")
    ap.add_argument("--no-dropin", action="store_true", help="skip the Parallel_env (reference-typed) call measurement")
    ap.add_argument("--no-train", action="store_true", help="skip the rollout + PPO update measurement")
    ap.add_argument("--no-workloads", action="store_true", help="skip the J10M10E3 / J30M20E5 lines")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (a fixed, seeded sample of rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
