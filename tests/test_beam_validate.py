"""Beam-search validation (validate.beam_validate): the selection rule against a brute force, the whole search against a
gather-free beam search that rebuilds every beam by replaying its action prefix on a fresh env batch, independence of
an instance's result from the chunking and from the other instances, and every returned schedule replayed on a fresh
env."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

GOLD = os.path.join(os.path.dirname(__file__), "golden")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")

WEIGHTS = (0.4, 0.4, 0.2)


def _brute_select(score, W):
    """Slot w takes the child of rank w under (score descending, flat index ascending); a -inf child makes the slot dead
    and it takes the rank-0 child."""
    S, C = score.shape
    child, slot, alive = np.zeros((S, W), np.int64), np.zeros((S, W)), np.zeros((S, W), bool)
    for s in range(S):
        ranked = sorted(range(C), key=lambda c: (-score[s, c], c))
        for w in range(W):
            c = ranked[w]
            alive[s, w] = score[s, c] > -np.inf
            child[s, w] = c if alive[s, w] else ranked[0]
            slot[s, w] = score[s, c]
    return child, slot, alive


@pytest.mark.parametrize("W", [1, 3, 8])
def test_selection_rule_matches_a_brute_force(W):
    rng = np.random.default_rng(W)
    S, C = 40, 72
    score = np.round(rng.normal(size=(S, C)), 1)  # one decimal: many exact ties
    score[rng.random((S, C)) < 0.4] = -np.inf
    score[:5] = -np.inf                            # instances without a single finite child ...
    score[5:10, :] = -np.inf                       # ... and with fewer finite children than slots
    score[5:10, rng.integers(0, C, 5)] = 0.5
    score[10:12] = 1.25                            # all tied
    child, slot, alive = val.beam_select(torch.as_tensor(score), W)
    bc, bs, ba = _brute_select(score, W)
    np.testing.assert_array_equal(child.numpy(), bc)
    np.testing.assert_array_equal(slot.numpy(), bs)
    np.testing.assert_array_equal(alive.numpy(), ba)


def _shipped(n=None):
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    return g, {k: pd[k][:n] for k in ("t", "p", "transT", "edge")}


def _objective(final4):
    w = WEIGHTS
    return w[0] * final4[..., 0] + w[1] * (final4[..., 1] + final4[..., 3]) + w[2] * final4[..., 2]


def _gather_free_beam(job, mch, inst, W):
    """Beam search without the gather: every step rebuilds each beam's env by loading, resetting and replaying its action
    prefix on one fresh env batch of the beam search's shape, runs the same actor calls at the same shapes, and selects
    with the brute force above.  -> actions [N,S*W,2] (env s*W + w), log_prob [S,W], final4 [S,W,4]."""
    S, N, M = inst["t"].shape
    J, E, B = N // M, inst["edge"].shape[1], S * W
    rep = {k: np.repeat(inst[k], W, axis=0) for k in ("t", "p", "transT", "edge")}
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)

    def rebuild(prefix):
        env.load(rep["t"], rep["p"], rep["transT"], rep["edge"])
        env.scaler_init()
        env.reset(np.tile(np.asarray(WEIGHTS), (B, 1)))
        env.obs(envm.MASK_ESA)
        for a in prefix:
            t = torch.as_tensor(a, device="cuda")
            env.step_obs(t[:, 0].contiguous(), t[:, 1].contiguous(), envm.MASK_ESA)

    prefix = np.zeros((0, B, 2), np.int32)
    score = np.full((S, W), -np.inf)
    score[:, 0] = 0.0
    h = None
    with torch.no_grad():
        for step in range(N):
            rebuild(prefix)
            pj, pooled, _ = job.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, h, env.job_mask, groups=B)
            f1, mm = [], []
            for j in range(J):
                a, b = env.mfea1(env.candidate[:, j].contiguous())
                f1.append(a.clone())
                mm.append(b.clone())
            f1 = torch.stack(f1, 1).view(B * J, M, -1)
            mm = torch.stack(mm, 1).view(B * J, M)
            pm, hm, _ = mch.forward(f1, env.mach_fea.repeat_interleave(J, 0), pooled.repeat_interleave(J, 0), mm, groups=B * J)
            lj = torch.log(pj).double().cpu().numpy().reshape(B, J, 1)
            lm = torch.log(pm).double().cpu().numpy().reshape(B, J, M)
            bad = env.job_mask.cpu().numpy().astype(bool).reshape(B, J, 1) | mm.cpu().numpy().astype(bool).reshape(B, J, M)
            with np.errstate(invalid="ignore"):
                child = (score.reshape(B, 1, 1) + lj) + lm
            child = np.where(bad, -np.inf, child).reshape(S, W * J * M)
            pick, score, _ = _brute_select(child, W)
            parent = (np.arange(S)[:, None] * W + pick // (J * M)).reshape(-1)
            jj = ((pick // M) % J).reshape(-1)
            cand = env.candidate.cpu().numpy()
            act = np.stack((cand[parent, jj], (pick % M).reshape(-1)), axis=1).astype(np.int32)
            prefix = np.concatenate((prefix[:, parent], act[None]), axis=0)
            h = hm.index_select(0, torch.as_tensor(parent * J + jj, device="cuda"))
    rebuild(prefix)
    assert env.done.cpu().numpy().all() and not env.invalid.cpu().numpy().any()
    return prefix, score, env.costs().cpu().numpy().reshape(S, W, 4)


def _check_against_reference(job, mch, inst, W):
    S, N = inst["t"].shape[:2]
    out = val.beam_validate(job, mch, inst, W, return_actions=True)
    acts, lp, f4 = _gather_free_beam(job, mch, inst, W)
    np.testing.assert_array_equal(out["actions"], acts.reshape(N, S, W, 2).transpose(0, 2, 1, 3))
    np.testing.assert_array_equal(out["log_prob"], lp.T)
    np.testing.assert_array_equal(out["final4"], f4.transpose(1, 0, 2))
    obj = np.where(lp.T > -np.inf, _objective(f4.transpose(1, 0, 2)), np.inf)
    np.testing.assert_array_equal(out["best_index"], obj.argmin(axis=0))
    assert out["alive"].all(axis=0).any()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tf32", "fp32"])
def test_beam_equals_a_gather_free_beam_search_on_shipped_instances(precision):
    g, inst = _shipped(8)
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    _check_against_reference(enc.JobActor(sd_op, 6, 6, precision=precision), enc.MachineActor(sd_m, 6, precision=precision),
                             inst, 4)


@pytest.mark.gpu
def test_beam_equals_a_gather_free_beam_search_two_tiles_per_env():
    J, M, E, S = 15, 10, 2, 3  # N = 150: two 128-row tiles per env on the grouped tcgen05 encoder
    d = ins.synthetic_instances(0, S, J, M, E, 515)
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(), 7), J, M, precision="tf32")
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(), 8), M, precision="tf32")
    _check_against_reference(job, mch, {k: d[k] for k in ("t", "p", "transT", "edge")}, 3)


def _replay(inst, actions, final4):
    """actions [N,W,S,2] on a fresh env batch (env w * S + s) -> every final4 bit for bit, no invalid env."""
    N, W, S, _ = actions.shape
    rep = {k: np.tile(inst[k], (W,) + (1,) * (inst[k].ndim - 1)) for k in ("t", "p", "transT", "edge")}
    env = envm.BatchedMTFJSPEnv(W * S, 6, 6, 2, obs_dtype=torch.float32)
    env.load(rep["t"], rep["p"], rep["transT"], rep["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(WEIGHTS), (W * S, 1)))
    a = torch.as_tensor(actions.reshape(N, W * S, 2), device="cuda")
    for step in range(N):
        env.step(a[step, :, 0].contiguous(), a[step, :, 1].contiguous())
        assert not env.invalid.cpu().numpy().any()
    assert env.done.cpu().numpy().all()
    np.testing.assert_array_equal(env.costs().cpu().numpy(), final4.reshape(W * S, 4))


@pytest.mark.gpu
def test_instance_results_do_not_depend_on_chunking_or_position_and_replay():
    g, inst = _shipped()
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    job, mch = enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32")
    W, S = 4, 100
    one = val.beam_validate(job, mch, inst, W, return_actions=True)
    small = val.beam_validate(job, mch, inst, W, max_envs=28, return_actions=True)  # 7 instances per chunk, a short last one
    keys = ("final4", "log_prob", "alive", "objective", "best_index", "best_final4", "actions", "best_actions")
    for k in keys:
        np.testing.assert_array_equal(small[k], one[k], err_msg=k)
    for s in range(S):
        alone = val.beam_validate(job, mch, {k: v[s:s + 1] for k, v in inst.items()}, W, return_actions=True)
        for k in ("final4", "log_prob", "alive", "objective", "actions"):
            np.testing.assert_array_equal(alone[k][..., 0, :] if k in ("final4", "actions") else alone[k][:, 0],
                                          one[k][..., s, :] if k in ("final4", "actions") else one[k][:, s],
                                          err_msg="instance %d: %s" % (s, k))
        assert alone["best_index"][0] == one["best_index"][s]
    # every returned schedule, and the best ones, replayed on a fresh env
    _replay(inst, one["actions"], one["final4"])
    _replay(inst, one["best_actions"][:, None], one["best_final4"][None])
    np.testing.assert_array_equal(one["objective"], _objective(one["final4"]))
    obj = np.where(one["alive"], one["objective"], np.inf)
    np.testing.assert_array_equal(one["best_index"], obj.argmin(axis=0))
    np.testing.assert_array_equal(one["best_objective"], obj.min(axis=0))
    assert one["alive"][0].all()
