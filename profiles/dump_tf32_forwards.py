"""Seeded tf32 actor forwards and a seeded rollout, saved for a bitwise comparison of two builds of the library:

    python profiles/dump_tf32_forwards.py OUT.npz            # run on one tree
    python profiles/dump_tf32_forwards.py --compare A.npz B.npz [C.npz ...]

Forwards of JobActor, MachineActor and EsaMachineActor (tf32, return_logits) on live env states:
    J6M6E2, 4,096 envs, BatchNorm groups 1, 64 and 4,096 (one env per group; the tf32 ESA actor takes one group only);
    J30M20E5, 256 envs (N = 600 > 128: the aggregation + layer fallback of the job encoder).
Then 20 steps of a sampled `Rollout` (J6M6E2, 4,096 envs, seed 3): actions, log-probabilities, values and rewards.
--compare prints, per array, whether it is bit-identical across the files and the largest absolute difference from the
first file."""
import importlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def env_state(J, M, E, B, seed, steps=3):
    import torch
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed))
    env.obs(envm.MASK_ESA)
    for _ in range(steps):
        env.random_step(seed=seed, env_offset=0)
        env.obs(envm.MASK_ESA)
    return env, ins.random_weights(0, B, seed)


def forwards(out, tag, J, M, E, B, groups_list):
    import torch
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    env, _ = env_state(J, M, E, B, seed=J * 100 + M)
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M, precision="tf32")
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, precision="tf32")
    esa = enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 22), M, precision="tf32")
    h_m = torch.randn((B, 128), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
    with torch.no_grad():
        for groups in groups_list:
            k = "%s_g%d_" % (tag, groups)
            s, pooled, jv = job.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, h_m, env.job_mask, groups=groups,
                                         return_logits=True)
            out[k + "job_scores"], out[k + "job_pooled"], out[k + "job_v"] = s, pooled, jv
            m1, mmask = env.mfea1(env.candidate[:, 0].contiguous())
            s, pooled, mv = mch.forward(m1, env.mach_fea, h_m, mmask, groups=groups, return_logits=True)
            out[k + "mch_scores"], out[k + "mch_pooled"], out[k + "mch_v"] = s, pooled, mv
            if groups == 1:
                s, pooled, mv = esa.forward(m1, env.mach_fea, h_m, mmask, return_logits=True)
                out[k + "esa_scores"], out[k + "esa_pooled"], out[k + "esa_v"] = s, pooled, mv


def rollout(out, steps=20):
    import torch
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
    J, M, E, B = 6, 6, 2, 4096
    env, w = env_state(J, M, E, B, seed=3, steps=0)
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M, precision="tf32")
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, precision="tf32")
    ro = rom.Rollout(env, job, mch, greedy=False, seed=3)
    ro.begin_episode(w)
    for t in range(steps):
        ro.step()
        for name, v in (("op", env.op), ("mach", env.mach), ("log_a", ro.log_a), ("m_log_a", ro.m_log_a),
                        ("job_v", ro.job_v), ("mch_v", ro.mch_v), ("reward5", env.reward5), ("task_fea", env.task_fea)):
            out["rollout_%02d_%s" % (t, name)] = v.clone()


def dump(path):
    import torch
    out = {}
    forwards(out, "J6M6", 6, 6, 2, 4096, (1, 64, 4096))
    forwards(out, "J30M20", 30, 20, 5, 256, (1,))
    rollout(out)
    torch.cuda.synchronize()
    np.savez(path, **{k: v.detach().cpu().numpy() for k, v in out.items()})
    print("wrote %d arrays to %s" % (len(out), path))


def compare(paths):
    files = [np.load(p) for p in paths]
    same = 0
    for k in files[0].files:
        arrs = [f[k] for f in files]
        if all(np.array_equal(arrs[0], a, equal_nan=True) for a in arrs[1:]):
            same += 1
            continue
        dev = [float(np.nanmax(np.abs(a.astype(np.float64) - arrs[0].astype(np.float64)))) for a in arrs[1:]]
        print("%-28s differs; max |x - x[%s]|: %s" % (k, os.path.basename(paths[0]),
                                                      ", ".join("%s %.3g" % (os.path.basename(p), d) for p, d in zip(paths[1:], dev))))
    print("%d / %d arrays bit-identical across %s" % (same, len(files[0].files), ", ".join(map(os.path.basename, paths))))


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        compare(sys.argv[2:])
    else:
        dump(sys.argv[1])
