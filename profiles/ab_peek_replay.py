"""A/B timing of the one-step lookahead and the whole-episode replay between two builds of the library
(profiles/README.md, "Lookahead and replay on the step's shared device code").

  python profiles/ab_peek_replay.py OUT.json LIB_A LIB_B [ROUNDS]

Each round runs one child process per build, A then B, with MTFJSP_LIB pointing at that build.  A child measures
  peek    mtfjsp_peek of every (candidate op, machine) pair (K = J*M) mid-episode at the three sizes of prof_peek.py (a),
          with its setup and timing: L2 overwritten before every call, median of 20 after 3 untimed calls;
  replay  mtfjsp_replay of complete random-rollout sequences at the three sizes of prof_local_search.py (a), with its
          setup and timing: L2 overwritten before every call, median of 10 after 2 untimed calls;
and reports the medians and a SHA-256 of every output.  The parent process reports per build the median and the range
of the round medians, and whether every output hash agrees across builds and rounds."""
import hashlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def child():
    import numpy as np
    import torch

    sys.path.insert(0, HERE)
    import prof_local_search as pls
    import prof_peek as pp

    lib = pp.envm._lib.lib()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    s = pp.C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {"device": torch.cuda.get_device_name(0), "peek": {}, "replay": {}}
    for B, J, M, E in pp.SIZES:
        env = pp.mid_episode(B, J, M, E)
        K = J * M
        op = env.candidate_ops().unsqueeze(2).expand(B, J, M).reshape(B, K).contiguous()
        mach = torch.arange(M, dtype=torch.int32, device=env.device).repeat(J).expand(B, K).contiguous()
        r5 = torch.empty((B, K, 5), dtype=torch.float64, device=env.device)
        inv = torch.empty((B, K), dtype=torch.uint8, device=env.device)
        call = lambda: pp.envm.check(lib.mtfjsp_peek(env._h, pp.ptr(op), pp.ptr(mach), K, pp.ptr(r5), pp.ptr(inv), s),
                                     "mtfjsp_peek")
        for _ in range(3):
            call()
        t = [pp.ev_time(call, flush) for _ in range(20)]
        out["peek"]["J%dM%d" % (J, M)] = {"envs": B, "K": K, "s": float(np.median(t)), "sha256": digest(r5, inv)}
        env.close()
    for B, J, M, E in pls.SIZES:
        N = J * M
        d = pls.ins.device_instances(0, B, J, M, E, seed=91)
        env = pls.fresh_env(d, pls.ins.random_weights(0, B, 91), B, J, M, E)
        acts = []
        for _ in range(N):
            env.random_step(seed=13)
            acts.append(torch.stack((env.op, env.mach), 1).clone())
        act = torch.stack(acts).transpose(0, 1).contiguous()  # [B,N,2]
        src = torch.arange(B, dtype=torch.int32, device=env.device)
        f4 = torch.empty((B, 4), dtype=torch.float64, device=env.device)
        r5 = torch.empty((B, 5), dtype=torch.float64, device=env.device)
        fi = torch.empty((B,), dtype=torch.int32, device=env.device)
        call = lambda: pls.envm.check(lib.mtfjsp_replay(env._h, pls.ptr(src), B, pls.ptr(act), N, pls.ptr(f4),
                                                        pls.ptr(r5), pls.ptr(fi), s), "mtfjsp_replay")
        for _ in range(2):
            call()
        t = [pls.ev_time(call, flush) for _ in range(10)]
        out["replay"]["J%dM%d" % (J, M)] = {"envs": B, "T": N, "s": float(np.median(t)), "sha256": digest(f4, r5, fi)}
        env.close()
    print(json.dumps(out))


def main():
    out_path, libs = sys.argv[1], {"A": os.path.abspath(sys.argv[2]), "B": os.path.abspath(sys.argv[3])}
    rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    runs = {k: [] for k in libs}
    for _ in range(rounds):
        for k, path in libs.items():
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], capture_output=True, text=True,
                               env=dict(os.environ, MTFJSP_LIB=path))
            if r.returncode != 0:
                sys.exit("child (%s) failed:\n%s" % (path, r.stderr))
            runs[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
    res = {"nvidia_smi name,power.limit,clocks.max.sm": smi, "libs": libs, "rounds": rounds, "table": {}}
    hashes_equal = True
    for kind in ("peek", "replay"):
        for size in runs["A"][0][kind]:
            row = {}
            for k in libs:
                ts = sorted(run[kind][size]["s"] for run in runs[k])
                row[k] = {"median_ms": 1e3 * ts[len(ts) // 2], "min_ms": 1e3 * ts[0], "max_ms": 1e3 * ts[-1],
                          "runs_ms": [1e3 * run[kind][size]["s"] for run in runs[k]]}
            hs = {run[kind][size]["sha256"] for k in libs for run in runs[k]}
            row["outputs_equal"] = len(hs) == 1
            hashes_equal &= row["outputs_equal"]
            res["table"]["%s %s" % (kind, size)] = row
    res["outputs_equal"] = hashes_equal
    res["device"] = runs["A"][0]["device"]
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    child() if sys.argv[1:] == ["--child"] else main()
