"""Overlapped step launches (MTFJSP_LAUNCH_OVERLAP, default on: a whole-batch step launch may start while the previous
one finishes, each warp waiting for its own envs) against plain stream order (MTFJSP_LAUNCH_OVERLAP=0).  Steps are
issued back to back without host synchronisation, at batch sizes of more than one wave of resident blocks, so that
J6M6 launches do overlap; at the other sizes (which launch in stream order) the switch must change nothing.  Every
call sequence must leave byte-identical outputs and state on both settings, and no launch may time out waiting
(launch_overlap_error stays 0)."""
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")

# (J, M, E, B): several waves of the size's specialised kernel; J30M20 is a COLD kernel
SIZES = [(6, 6, 2, 20011), (10, 10, 3, 8191), (30, 20, 5, 2049)]
OUT = ["op", "mach", "mfea1_buf", "mach_mask", "reward5", "scaled4", "done", "invalid", "task_fea", "mach_fea", "adj_w",
       "adj_src", "job_mask", "candidate"]


def snapshot(env):
    out = {n: getattr(env, n).cpu().numpy().copy() for n in OUT}
    out.update({"st_" + k: v.cpu().numpy() for k, v in env.export_state().items()})
    out.update({"sc_" + k: v.cpu().numpy() for k, v in env.export_scaler().items()})
    out["costs"] = env.costs().cpu().numpy()
    assert env.launch_overlap_error == 0
    return out


def make_env(size, seed=21):
    J, M, E, B = size
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    return env, torch.as_tensor(ins.random_weights(0, B, seed), device="cuda")


def random_episodes(size):
    env, w = make_env(size)
    rec = []
    env.reset(w)
    for _ in range(env.N):
        env.random_step(seed=3, env_offset=11)
    rec.append(snapshot(env))
    env.reset(w)
    env.scaler_reset()
    for _ in range(env.N // 2):
        env.random_step(seed=4, env_offset=0)
    rec.append(snapshot(env))
    return rec


def recorded_actions(size):
    """step_obs replaying the actions of a random episode, from a device array (no other launch between the steps)"""
    env, w = make_env(size)
    env.reset(w)
    ops, machs = [], []
    for _ in range(env.N):
        env.random_step(seed=7, env_offset=5)
        ops.append(env.op.clone())
        machs.append(env.mach.clone())
    acts_op, acts_mach = torch.stack(ops), torch.stack(machs)
    env.reset(w)
    env.scaler_reset()
    env.obs()
    for s in range(env.N):
        env.step_obs(acts_op[s], acts_mach[s])
    return [snapshot(env)]


def fused_reset_mid_episode(size):
    env, w = make_env(size)
    w2 = torch.as_tensor(ins.random_weights(0, env.B, 22), device="cuda")
    env.reset(w)
    for _ in range(5):
        env.random_step(seed=3, env_offset=11)
    env.reset(w2)  # recorded: the next step launch performs it
    env.scaler_reset()
    for _ in range(env.N // 2):
        env.random_step(seed=3, env_offset=11)
    return [snapshot(env)]


def host_and_foreign_between(size):
    env, w = make_env(size)
    env.reset(w)
    for _ in range(3):
        env.random_step(seed=3, env_offset=11)
    env.policy_random(seed=9)
    acts = torch.stack([env.op.cpu(), env.mach.cpu()], 1).contiguous().pin_memory()
    recs = env.host_buffers()[1]
    env.random_step(seed=3, env_offset=11)
    env.step_host_packed(acts, recs)  # the host-step kernel between two step launches
    env.random_step(seed=3, env_offset=11)
    acc = torch.zeros(1, dtype=torch.float64, device="cuda")
    for _ in range(4):
        env.random_step(seed=3, env_offset=11)
        acc += env.reward5[:, 0].sum()  # a foreign kernel reading the previous step's output
    rec = snapshot(env)
    rec["records"] = recs.numpy().copy()
    rec["acc"] = acc.cpu().numpy()
    return [rec]


def two_handles(size):
    a, wa = make_env(size, 21)
    b, wb = make_env(size, 31)
    a.reset(wa)
    b.reset(wb)
    for s in range(a.N):
        a.random_step(seed=3, env_offset=11)
        b.random_step(seed=5, env_offset=0)
        if s % 3 == 0:
            a.random_step(seed=3, env_offset=11)
    return [snapshot(a), snapshot(b)]


def own_actions_and_scaler_reset(size):
    """a step fed the action the previous random step drew, and a scaler reset alone, between random steps"""
    env, w = make_env(size)
    env.reset(w)
    for s in range(env.N // 2):
        env.random_step(seed=3, env_offset=11)
        if s % 4 == 1:
            env.step_obs(env.op, env.mach)  # already scheduled: every env reports it invalid
        if s == 7:
            env.scaler_reset()
    return [snapshot(env)]


CASES = {"random_episodes": random_episodes, "recorded_actions": recorded_actions,
         "fused_reset_mid_episode": fused_reset_mid_episode, "host_and_foreign_between": host_and_foreign_between,
         "two_handles": two_handles, "own_actions_and_scaler_reset": own_actions_and_scaler_reset}


def compare(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.keys() == w.keys()
        for k in w:
            np.testing.assert_array_equal(g[k], w[k], err_msg="record %d, %s" % (i, k))


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%d" % s[:2])
def test_overlapped_launches_match_stream_order(size, case, monkeypatch):
    if case in ("recorded_actions", "host_and_foreign_between", "two_handles", "own_actions_and_scaler_reset") and \
            size[0] != 6:
        pytest.skip("J6M6 only")
    res = {}
    for setting in ("0", "1"):
        monkeypatch.setenv("MTFJSP_LAUNCH_OVERLAP", setting)
        res[setting] = CASES[case](size)
        torch.cuda.synchronize()
    compare(res["1"], res["0"])


def test_cuda_graph_rollout_matches_stream_order(monkeypatch):
    """rollout.Rollout replaying one CUDA graph per step: the captured step launches take no part in the overlap"""
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    ro_mod = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
    J, M = 6, 6
    res = {}
    for setting in ("0", "1"):
        monkeypatch.setenv("MTFJSP_LAUNCH_OVERLAP", setting)
        env, w = make_env((J, M, 2, 4099))
        job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 11), J, M)
        mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M)
        ro = ro_mod.Rollout(env, job, mch, greedy=True, use_cuda_graph=True)
        c1 = ro.run_episode(w).cpu().numpy()
        for _ in range(4):  # eager step launches behind the graph replays
            env.random_step(seed=3, env_offset=0)
        c2 = ro.run_episode(w).cpu().numpy()
        res[setting] = [{"c1": c1, "c2": c2, **snapshot(env)}]
    compare(res["1"], res["0"])
