"""mtfjsp_replay / BatchedMTFJSPEnv.replay: the costs, summed rewards and first invalid index of whole action sequences
replayed from an env's episode start, without changing the env.  Checked bit for bit against a fresh copy of the env
taken right after its reset (gather_from) and stepped with the same actions, at the sizes of test_env_peek (specialised,
unspecialised, N > 128 and the size edges), with and without left shift, at T = 1, N/2 and N, with more candidates than
envs and duplicated / permuted sources; with invalid actions mid-sequence; after recorded resets and gathers; and
against the final costs greedy validation, beam search and GREEDY_R report.  A twin handle that never replays shows
that nothing of the env is written."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
from tests.test_env_peek import OUT, SIZES  # noqa: E402

E_ARG, E_STATE = -1, -3
GOLD = os.path.join(os.path.dirname(__file__), "golden")
B = 6


def _make(J, M, E, left_shift, d, w, B_=B):
    env = envm.BatchedMTFJSPEnv(B_, J, M, E, left_shift=left_shift, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    env.obs()
    return env


def _data(J, M, E, seed, B_=B):
    return ins.synthetic_instances(0, B_, J, M, E, seed=seed), ins.random_weights(0, B_, seed=seed)


def _random_episode(env, seed):
    """Steps env through a whole random episode; returns its actions [N,B,2] int32."""
    acts = []
    for _ in range(env.N):
        env.random_step(seed=seed)
        acts.append(torch.stack((env.op, env.mach), 1).clone())
    return torch.stack(acts)


def _composed(fresh, src, acts, left_shift):
    """What replay must return: copies of fresh's envs src (fresh is at its episode start), stepped with acts [T,R,2],
    rewards summed in step order from 0.0, costs, and the first step whose invalid flag is set."""
    T, R, _ = acts.shape
    cp = envm.BatchedMTFJSPEnv(R, fresh.J, fresh.M, fresh.E, left_shift=left_shift, obs_dtype=torch.float32)
    cp.gather_from(fresh, src)
    tot = torch.zeros((R, 5), dtype=torch.float64, device=cp.device)
    first = torch.full((R,), -1, dtype=torch.int32, device=cp.device)
    for s in range(T):
        cp.step(acts[s, :, 0].contiguous(), acts[s, :, 1].contiguous())
        tot += cp.reward5
        first = torch.where((first < 0) & (cp.invalid != 0), s, first)
    out = cp.costs(), tot, first
    cp.close()
    return out


def _assert_equal(got, exp, where):
    for name, g, e in zip(("final4", "return5", "first_invalid"), got, exp):
        np.testing.assert_array_equal(g.cpu().numpy(), e.cpu().numpy(), err_msg="%s %s" % (where, name))


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_replay_equals_steps(size, left_shift):
    J, M, E = size
    N = J * M
    d, w = _data(J, M, E, 40 + J)
    env = _make(J, M, E, left_shift, d, w)
    fresh = _make(J, M, E, left_shift, d, w)
    acts = _random_episode(env, seed=3)                                       # env ends the episode: replay starts over
    dev = env.device
    src = torch.tensor([5, 0, 0, 3, 1, 2, 4, 5, 2, 1, 3], dtype=torch.int32, device=dev)   # R > B, duplicated, permuted
    seqs = acts.index_select(1, src.long())
    for T in sorted({1, N // 2, N}):
        got = env.replay(seqs[:T], src)
        _assert_equal(got, _composed(fresh, src, seqs[:T], left_shift), "T=%d" % T)
        assert (got[2] == -1).all()
    got = env.replay(acts)                                                    # src=None: env r from row r
    _assert_equal(got, _composed(fresh, torch.arange(B, dtype=torch.int32, device=dev), acts, left_shift), "src=None")
    np.testing.assert_array_equal(got[0].cpu().numpy(), env.costs().cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (30, 20, 5), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_invalid_actions_are_no_ops_and_reported(size):
    J, M, E = size
    N = J * M
    d, w = _data(J, M, E, 7)
    env = _make(J, M, E, True, d, w)
    fresh = _make(J, M, E, True, d, w)
    acts = _random_episode(env, seed=9)
    dev = env.device
    t = torch.as_tensor(d["t"], device=dev)
    src = torch.arange(B, dtype=torch.int32, device=dev).repeat(8)
    seqs = acts.index_select(1, src.long()).clone()
    s0 = N // 3
    ar = torch.arange(seqs.shape[1], device=dev)
    kind = ar // B
    op, mc = seqs[s0, :, 0].clone(), seqs[s0, :, 1].clone()
    infeas = torch.where((t[src.long(), op.long()] < 0).any(1), (t[src.long(), op.long()] < 0).int().argmax(1), M)
    bad_op = torch.stack((seqs[0, :, 0], op + 1, op, torch.full_like(op, N), torch.full_like(op, -1), op, op, op))[kind, ar]
    bad_m = torch.stack((seqs[0, :, 1], mc, infeas.to(torch.int32), mc, mc, torch.full_like(mc, M), torch.full_like(mc, -1),
                         mc))[kind, ar]
    # 0 an already scheduled op, 1 a skipped job predecessor (may be valid at a job's last op), 2 an infeasible machine
    # (or M where every machine is feasible), 3-6 out-of-range op / machine, 7 unchanged (then step s0 + 1 repeats it, an
    # already scheduled op); the sequence goes on after it
    ins_ = torch.cat((seqs[:s0], torch.stack((bad_op, bad_m), 1)[None], seqs[s0:N - 1]))
    got = env.replay(ins_, src)
    _assert_equal(got, _composed(fresh, src, ins_, True), "invalid")
    fi = got[2].cpu().numpy()
    k = kind.cpu().numpy()
    assert (fi[(k == 0) | (k >= 2) & (k <= 6)] == s0).all() and (fi[k == 7] == s0 + 1).all()


def _state(env):
    st = env.export_state()
    sc = env.export_scaler()
    return [x.cpu().numpy() for x in list(st.values()) + list(sc.values()) + [env.costs()]]


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (10, 10, 3), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_replay_leaves_the_env_untouched(size):
    J, M, E = size
    N = J * M
    d, w = _data(J, M, E, 17)
    a = _make(J, M, E, True, d, w)
    b = _make(J, M, E, True, d, w)
    ref = _make(J, M, E, True, d, w)
    acts = _random_episode(ref, seed=4)
    for s in range(N - 2):
        if s % 3 == 0:
            idx = torch.tensor([1, 1, 0, 5, 2], dtype=torch.int32, device=a.device).repeat(3)
            a.replay(acts[: 1 + s].index_select(1, idx.long()), idx)
        op, mc = acts[s, :, 0].contiguous(), acts[s, :, 1].contiguous()
        a.step_obs(op, mc)
        b.step_obs(op, mc)
        for x, y, n in zip([getattr(a, k) for k in OUT], [getattr(b, k) for k in OUT], OUT):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg="step %d %s" % (s, n))
    for x, y in zip(_state(a), _state(b)):
        np.testing.assert_array_equal(x, y)
    a.replay(acts)
    for e in (a, b):  # overlapped back-to-back steps after a replay
        e.random_step(seed=1)
        e.random_step(seed=1)
    torch.cuda.synchronize()
    for x, y, n in zip([getattr(a, k) for k in OUT], [getattr(b, k) for k in OUT], OUT):
        np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg=n)
    for x, y in zip(_state(a), _state(b)):
        np.testing.assert_array_equal(x, y)
    a.check_launch_overlap()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"])
def test_replay_after_recorded_reset_and_on_a_gather_destination(fused, monkeypatch):
    monkeypatch.setenv("MTFJSP_FUSED_RESET", fused)
    J, M, E = 6, 6, 2
    d, w = _data(J, M, E, 23)
    env = _make(J, M, E, True, d, w)
    fresh = _make(J, M, E, True, d, w)
    acts = _random_episode(env, seed=6)
    env.reset(w[::-1].copy())                                                  # recorded reset, then replay
    got = env.replay(acts)
    _assert_equal(got, _composed(fresh, torch.arange(B, dtype=torch.int32, device=env.device), acts, True), "reset")
    env.step(acts[0, :, 0].contiguous(), acts[0, :, 1].contiguous())           # the reset was performed before the step
    np.testing.assert_array_equal(env.export_state()["mach"].cpu().numpy() >= 0,
                                  (torch.arange(env.N, device=env.device)[None] == acts[0, :, :1]).cpu().numpy())
    idx = torch.tensor([3, 3, 1, 0, 5, 2, 4], dtype=torch.int32, device=env.device)
    dst = envm.BatchedMTFJSPEnv(7, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    dst.gather_from(env, idx)
    src = torch.tensor([6, 0, 2, 2], dtype=torch.int32, device=env.device)
    seqs = acts.index_select(1, idx[src.long()].long())
    _assert_equal(dst.replay(seqs, src), env.replay(seqs, idx[src.long()]), "gather")


@pytest.mark.gpu
def test_errors_write_nothing_and_bad_sources_are_rows_of_zeros():
    J, M, E = 6, 6, 2
    N = J * M
    d, w = _data(J, M, E, 29)
    lib = libm.lib()
    dev = torch.device("cuda", torch.cuda.current_device())
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    acts = torch.zeros((N, B, 2), dtype=torch.int32, device=dev)
    src = torch.arange(B, dtype=torch.int32, device=dev)
    c4 = torch.full((B, 4), 7.0, dtype=torch.float64, device=dev)
    r5 = torch.full((B, 5), 7.0, dtype=torch.float64, device=dev)
    fi = torch.full((B,), 7, dtype=torch.int32, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = env._h
    assert lib.mtfjsp_replay(h, p(src), B, p(acts), N, p(c4), p(r5), p(fi), st) == E_STATE   # loaded, never reset
    env.scaler_init()
    env.reset(w)
    for args in [(None, p(src), B, p(acts), N), (h, None, B, p(acts), N), (h, p(src), B, None, N), (h, p(src), 0, p(acts), N),
                 (h, p(src), B, p(acts), 0), (h, p(src), B, p(acts), N + 1)]:
        assert lib.mtfjsp_replay(*args, p(c4), p(r5), p(fi), st) == E_ARG
    torch.cuda.synchronize()
    assert (c4 == 7.0).all() and (r5 == 7.0).all() and (fi == 7).all()
    with pytest.raises(libm.MTFJSPError):
        env.replay(acts[:0])
    with pytest.raises(ValueError):
        env.replay(acts[:, :3])                                                # src=None needs R == B
    ref = _make(J, M, E, True, d, w)
    seq = _random_episode(ref, seed=2)
    bad = torch.tensor([0, -1, 2, B, 4, 1 << 30], dtype=torch.int32, device=dev)
    got = env.replay(seq, bad)
    good = env.replay(seq)
    ok = torch.tensor([True, False, True, False, True, False], device=dev)
    for g, e in zip(got, good):
        np.testing.assert_array_equal(g[ok].cpu().numpy(), e[ok].cpu().numpy())
        assert (g[~ok] == (-2 if g.dtype == torch.int32 else 0)).all()
    assert lib.mtfjsp_replay(h, p(src), B, p(seq.transpose(0, 1).contiguous()), N, None, None, None, st) == 0


@pytest.mark.gpu
def test_replay_reproduces_greedy_beam_and_greedy_r():
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
    rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k][:40] for k in ("t", "p", "transT", "edge")}
    S = 40
    op_sd, mch_sd = val.load_actor_state_dicts(os.path.join(GOLD, "policy_golden.npz"), "iotj")
    ja, ma = enc.JobActor(op_sd, 6, 6, precision="tf32"), enc.MachineActor(mch_sd, 6, precision="tf32")
    w = np.tile([0.4, 0.4, 0.2], (S, 1))
    for left_shift in (True, False):
        env = envm.BatchedMTFJSPEnv(S, 6, 6, 2, left_shift=left_shift, obs_dtype=torch.float32)
        env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
        env.scaler_init()
        env.reset(w)
        gr = val.greedy_validate(ja, ma, inst, left_shift=left_shift, return_actions=True)
        f4, r5, fi = env.replay(torch.as_tensor(gr["actions"], device=env.device))
        np.testing.assert_array_equal(f4.cpu().numpy(), gr["final4"])
        np.testing.assert_array_equal(r5.cpu().numpy(), gr["cumulative_rewards"])
        assert (fi == -1).all()
        bm = val.beam_validate(ja, ma, inst, 4, left_shift=left_shift, return_actions=True)
        f4, _, fi = env.replay(torch.as_tensor(bm["best_actions"], device=env.device))
        np.testing.assert_array_equal(f4.cpu().numpy(), bm["best_final4"])
        assert (fi == -1).all()
        env.reset(w)
        acts = rules.greedy_reward_rollout(env)
        f4, _, fi = env.replay(acts)
        np.testing.assert_array_equal(f4.cpu().numpy(), env.costs().cpu().numpy())
        assert (fi == -1).all()
        env.close()
