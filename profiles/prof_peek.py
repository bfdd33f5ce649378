"""One-step lookahead (profiles/README.md, "One-step lookahead").

  (a) mtfjsp_peek of every (candidate op, machine) pair (K = J*M) at 65,536 J6M6E2, 16,384 J10M10E3 and 4,096 J30M20E5
      envs, mid-episode (N/2 random steps, left shift on), through the C entry point into preallocated outputs: CUDA
      events around each call, L2 overwritten (256 MB memset) before every timed call, median of 20 calls after 3
      untimed ones.  Against the brute force producing the same arrays: mtfjsp_gather of every env into K copies, then
      mtfjsp_step of every copy, in chunks of at most CHUNK_BYTES of copy state; events around the whole chunked pass,
      median of 3 after 1 untimed one.  Both outputs (reward5, invalid) are compared for equality in the same run.
      Bytes: peek = mtfjsp_bytes_per_peek(K) x envs (records staged once per env, per pair its pair, t / p entries and
      outputs); brute force = (mtfjsp_bytes_per_gather + the step's record traffic, mtfjsp_bytes_per_step) x envs x K.
  (b) wall time of each new rule (LWKR_IT / MWKR_IT x SPT / SEC, GREEDY_R) on the 100 shipped J6M6E2 test instances and
      on 65,536 device-generated J6M6E2 instances: host clock around the rollout (ends in a device synchronise), median
      of 3 after one untimed rollout.
  (c) mean objective over the 100 shipped test instances of every evaluate_rules row (the ten static rows and the five
      new ones) and of greedy_validate with the shipped `iotj` checkpoint (tf32).
Prints the results as JSON and writes them to the path given as the first argument (default profiles/peek_b200.json)."""
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
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
GOLD = os.path.join(ROOT, "tests", "golden")
SIZES = [(65536, 6, 6, 2), (16384, 10, 10, 3), (4096, 30, 20, 5)]
CHUNK_BYTES = 24 << 30


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


def ev_time(fn, flush=None):
    if flush is not None:
        flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3


def ptr(x):
    return C.c_void_p(x.data_ptr())


def mid_episode(B, J, M, E):
    d = ins.device_instances(0, B, J, M, E, seed=77)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 77))
    env.obs()
    for _ in range(J * M // 2):
        env.random_step(seed=5)
    return env


def peek_vs_brute(B, J, M, E, flush):
    lib = envm._lib.lib()
    env = mid_episode(B, J, M, E)
    K = J * M
    op = env.candidate_ops().unsqueeze(2).expand(B, J, M).reshape(B, K).contiguous()
    mach = torch.arange(M, dtype=torch.int32, device=env.device).repeat(J).expand(B, K).contiguous()
    r5 = torch.empty((B, K, 5), dtype=torch.float64, device=env.device)
    inv = torch.empty((B, K), dtype=torch.uint8, device=env.device)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda: lib.mtfjsp_peek(env._h, ptr(op), ptr(mach), K, ptr(r5), ptr(inv), s)
    for _ in range(3):
        call()
    t_peek = [ev_time(call, flush) for _ in range(20)]
    # brute force: chunks of envs, each env copied K times and stepped once
    per_copy = int(lib.mtfjsp_bytes_per_gather(env._h)) + 8 * J * M * M * 2  # records + t / p tables held per copy
    Bc = max(1, min(B, CHUNK_BYTES // (per_copy * K)))
    cp = envm.BatchedMTFJSPEnv(Bc * K, J, M, E, obs_dtype=torch.float32)
    idx_all = torch.arange(B, dtype=torch.int32, device=env.device).repeat_interleave(K)
    opf, machf = op.reshape(-1), mach.reshape(-1)
    b5 = torch.empty((B * K, 5), dtype=torch.float64, device=env.device)
    binv = torch.empty((B * K,), dtype=torch.uint8, device=env.device)
    cp_r5 = torch.empty((Bc * K, 5), dtype=torch.float64, device=env.device)
    cp_inv = torch.empty((Bc * K,), dtype=torch.uint8, device=env.device)

    def brute():
        for c0 in range(0, B, Bc):
            n = min(Bc, B - c0) * K
            idx = idx_all[c0 * K:c0 * K + n]
            if n < Bc * K:  # last chunk: the spare copies duplicate env 0 and are not read
                idx = torch.cat((idx, torch.zeros(Bc * K - n, dtype=torch.int32, device=env.device)))
            o = torch.cat((opf[c0 * K:c0 * K + n], opf[:Bc * K - n])) if n < Bc * K else opf[c0 * K:c0 * K + n]
            m = torch.cat((machf[c0 * K:c0 * K + n], machf[:Bc * K - n])) if n < Bc * K else machf[c0 * K:c0 * K + n]
            envm.check(lib.mtfjsp_gather(cp._h, env._h, ptr(idx), s), "mtfjsp_gather")
            envm.check(lib.mtfjsp_step(cp._h, ptr(o), ptr(m), ptr(cp_r5), None, None, ptr(cp_inv), s), "mtfjsp_step")
            b5[c0 * K:c0 * K + n].copy_(cp_r5[:n])
            binv[c0 * K:c0 * K + n].copy_(cp_inv[:n])

    brute()
    t_brute = [ev_time(brute, flush) for _ in range(3)]
    same = bool(torch.equal(r5.reshape(-1, 5), b5) and torch.equal(inv.reshape(-1), binv))
    bp = int(lib.mtfjsp_bytes_per_peek(env._h, K)) * B
    bb = (int(lib.mtfjsp_bytes_per_gather(cp._h)) + int(lib.mtfjsp_bytes_per_step(cp._h, 0))) * B * K
    tp, tb = float(np.median(t_peek)), float(np.median(t_brute))
    out = {"envs": B, "J": J, "M": M, "E": E, "K": K, "pairs": B * K, "peek_s": tp, "peek_s_runs": t_peek,
           "brute_s": tb, "brute_s_runs": t_brute, "brute_chunk_envs": Bc, "brute_chunks": (B + Bc - 1) // Bc,
           "speedup": tb / tp, "outputs_equal": same, "peek_bytes": bp, "brute_bytes": bb,
           "peek_GBps": bp / tp / 1e9, "brute_GBps": bb / tb / 1e9,
           "valid_pairs": int((inv == 0).sum().item())}
    cp.close()
    env.close()
    return out


def rule_env(d, J, M, E):
    B = d["t"].shape[0]
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=False, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    w = np.tile([0.4, 0.4, 0.2], (B, 1))
    return env, w


def rule_times(d, tag):
    t_np = d["t"].cpu().numpy() if torch.is_tensor(d["t"]) else d["t"]
    p_np = d["p"].cpu().numpy() if torch.is_tensor(d["p"]) else d["p"]
    env, w = rule_env(d, 6, 6, 2)
    rows = []
    for name in ("LWKR_IT+SPT", "LWKR_IT+SEC", "MWKR_IT+SPT", "MWKR_IT+SEC", "GREEDY_R"):
        if name == "GREEDY_R":
            go = lambda: rules.greedy_reward_rollout(env)
        else:
            o, m = name.split("+")
            ml = torch.as_tensor(rules.machine_rule(m, t_np, p_np).astype(np.int32), device=env.device)
            go = lambda o=o, ml=ml: rules.lookahead_rollout(env, o, ml)

        def run():
            env.reset(w)
            return go()

        run()
        ts = [wall(run)[0] for _ in range(3)]
        ok = bool(env.done.all().item()) and not bool(env.invalid.any().item())
        rows.append({"instances": tag, "envs": env.B, "rule": name, "wall_s": float(np.median(ts)), "wall_s_runs": ts,
                     "per_decision_ms": float(np.median(ts)) / 36 * 1e3, "all_done_and_valid": ok})
        print(json.dumps(rows[-1]), flush=True)
    env.close()
    return rows


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "peek_b200.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info()}
    print(json.dumps(res["gpu"]), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res["peek"] = []
    for B, J, M, E in SIZES:
        res["peek"].append(peek_vs_brute(B, J, M, E, flush))
        print(json.dumps(res["peek"][-1]), flush=True)
    del flush
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    res["rules"] = rule_times(inst, "shipped_100") + rule_times(ins.device_instances(0, 65536, 6, 6, 2, seed=123), "device_65536")
    ev = rules.evaluate_rules(inst["t"], inst["p"], inst["transT"], inst["edge"], 6, 6, 2,
                              op_rules=rules.OP_RULES + rules.LOOKAHEAD_RULES, joint_rules=rules.JOINT_RULES)
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    greedy = val.greedy_validate(enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32"),
                                 inst, chunk=100)["objective"]
    res["quality"] = {"instances": "shipped_100", "mean_objective": {n: float(v.mean()) for n, v in zip(ev["names"], ev["objective"])}}
    res["quality"]["mean_objective"]["greedy_validate iotj tf32"] = float(greedy.mean())
    print(json.dumps(res["quality"], indent=1), flush=True)
    txt = json.dumps(res, indent=1)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(txt)


if __name__ == "__main__":
    main()
