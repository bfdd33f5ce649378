"""Measurements of end-to-end training (train.Trainer) and of the grouped machine trunk on the device.

usage: python profiles/prof_train_run.py MODE [--out FILE] [--episodes E]
  trunk       MachineActor tf32 forward at 65,536 J6M6 envs: groups = 4096 on the fused grouped trunk, groups = 4096 on the
              previous path (trunk kernel, separate grouped BatchNorm pass, head without input affine), groups = 1;
              alternated, CUDA events, plus the groups = 1 outputs (--dump FILE.npz) for byte comparison across builds
  learn       the short fixed-seed run of tests/test_train.py (G = 64): eval curve, FIFO+SPT on the same instances
  throughput  G = 512 (8,192 envs): training env-steps/s including evaluation
  reference   G = 1, the reference protocol (4,000 episodes unless --episodes): wall time and the eval curve
Each mode prints one JSON line (and writes it to --out) with the device name and power limit."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
tr = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.train")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return dict(device=torch.cuda.get_device_name(), nvidia_smi=q[0] if q else None)


class _PreviousGroupedTrunk(enc.MachineActor):
    """groups > 1 as before the grouped trunk kernel: trunk kernel, then a separate grouped BatchNorm pass over [B*M,128]."""

    def trunk(self, f1, f2, groups=1):
        w, H, M = self.w, self.H, self.M
        B = f1.shape[0]
        buf = enc.gat_trunk_tf32(f1.reshape(B * M, 6).contiguous(), f2.reshape(B * M, 8).contiguous(), w["m_fea_1_fcl.weight"],
                                 w["m_fea_2_fcl.weight"], self._derived("gat_Wt", lambda: w["gat_layer.W"].t()),
                                 self._derived("gat_a_src", lambda: w["gat_layer.a"][0, :H, 0]),
                                 self._derived("gat_a_dst", lambda: w["gat_layer.a"][0, H:, 0]))
        self._pending_m = None
        nodes = enc._bn_train(buf, w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, M, H)
        return nodes, nodes.mean(dim=1)


def trunk(args):
    B, J, M, E = 65536, 6, 6, 2
    g = torch.Generator("cuda").manual_seed(0)
    f1 = torch.rand(B, M, 6, device="cuda", generator=g) * 2 - 0.5
    f2 = torch.rand(B, M, 8, device="cuda", generator=g) * 2 - 0.5
    h_o = torch.randn(B, 128, device="cuda", generator=g) / 3
    mask = (torch.rand(B, M, device="cuda", generator=g) < 0.3).to(torch.uint8)
    mask[:, 0] = 0
    sd = enc.seeded_state_dict(enc.machine_actor_keys(128), 12)
    cur, prev = enc.MachineActor(sd, M, precision="tf32"), _PreviousGroupedTrunk(sd, M, precision="tf32")
    cases = [("fused_grouped_4096", cur, 4096), ("previous_grouped_4096", prev, 4096), ("groups_1", cur, 1)]
    out = {}
    with torch.no_grad():
        for name, net, G in cases:                                   # warm-up, and the outputs
            out[name] = [t.clone() for t in net.forward(f1, f2, h_o, mask, groups=G)]
        torch.cuda.synchronize()
        ms = {n: [] for n, _, _ in cases}
        reps = 50
        for _ in range(5):                                           # alternated rounds
            for name, net, G in cases:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    net.forward(f1, f2, h_o, mask, groups=G)
                e1.record()
                torch.cuda.synchronize()
                ms[name].append(e0.elapsed_time(e1) / reps)
    d = lambda a, b: float((a - b).abs().max())
    res = dict(mode="trunk", envs=B, M=M, ms_median={k: float(np.median(v)) for k, v in ms.items()},
               ms_min={k: float(np.min(v)) for k, v in ms.items()},
               prob_max_abs_diff_fused_vs_previous=d(out["fused_grouped_4096"][0], out["previous_grouped_4096"][0]),
               pooled_max_abs_diff_fused_vs_previous=d(out["fused_grouped_4096"][1], out["previous_grouped_4096"][1]))
    if args.dump:
        np.savez(args.dump, **{"groups_1_%d" % i: t.cpu().numpy() for i, t in enumerate(out["groups_1"])})
    return res


def run_trainer(cfg, fifo=False):
    t = tr.Trainer(cfg, log=lambda s: print(s, flush=True))
    t.run()
    res = dict(groups=cfg.groups, envs=cfg.groups * cfg.env_batch, episodes=cfg.episodes(), wall_s=t.wall_s,
               env_steps_per_s=t.env_steps / t.wall_s, eval_episode=[h["episode"] for h in t.history],
               eval_obj_mean=[h["obj_mean"] for h in t.history], last_eval=t.history[-1], updates=len(t.losses),
               final_losses=t.losses[-1][1] if t.losses else None)
    if fifo:
        e = t.eval_set
        res["fifo_spt_obj_mean"] = float(rules.evaluate_rules(e["t"], e["p"], e["transT"], e["edge"], 6, 6, 2, op_rules=("FIFO",),
                                                              machine_rules=("SPT",))["objective"][0].mean())
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=("trunk", "learn", "throughput", "reference"))
    ap.add_argument("--out")
    ap.add_argument("--dump")
    ap.add_argument("--episodes", type=int)
    ap.add_argument("--ckpt-dir", default=os.environ.get("TMPDIR", "/tmp"))
    a = ap.parse_args()
    torch.cuda.init()
    if a.mode == "trunk":
        res = trunk(a)
    elif a.mode == "learn":
        test = importlib.import_module("tests.test_train")
        res = dict(mode="learn", **run_trainer(tr.TrainConfig(out_dir=os.path.join(a.ckpt_dir, "learn"), **test.LEARN), fifo=True))
    elif a.mode == "throughput":
        res = dict(mode="throughput", **run_trainer(tr.TrainConfig(groups=512, episode_num=a.episodes or 50, n_train=8192,
                                                                   out_dir=os.path.join(a.ckpt_dir, "g512"))))
    else:
        res = dict(mode="reference", **run_trainer(tr.TrainConfig(groups=1, episode_num=a.episodes,
                                                                   out_dir=os.path.join(a.ckpt_dir, "g1")), fifo=True))
    res.update(device_info())
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
