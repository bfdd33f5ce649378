"""mtfjsp_complete / BatchedMTFJSPEnv.complete: what the rest of an episode costs when T forced actions and then a base
policy (random draws or a priority table) finish it from an env's current state, without changing the env.  Checked
bit for bit against the composition it restates -- a gather_from copy of the sources, T steps, then policy_random (or
the priority choice) and step until done -- at the sizes of test_env_peek, with and without left shift, under both job
masks and both bases, from the reset state and mid-episode, with invalid forced actions and duplicated / permuted
sources; against replay at T = N; and against the shipped rule rows (tests/golden/pdr_golden.npz) through
rules.priority_table.  On the CPU: the priority tables give back rules.op_rule's orders, and the argument errors."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")

E_ARG, E_STATE = -1, -3
PDR = os.path.join(os.path.dirname(__file__), "golden", "pdr_golden.npz")
SIZES = [(6, 6, 2), (10, 10, 3), (30, 20, 5), (13, 11, 3), (70, 2, 1), (2, 64, 4)]
B = 5


def _merge_by_key(key, J, M):
    """The order a priority completion schedules from the reset state under the FINISHED mask: at every step the job
    whose next op has the smallest key, ties to the lowest job."""
    S, N = key.shape
    out = np.zeros((S, N), dtype=np.int64)
    for s in range(S):
        nx = np.zeros(J, dtype=np.int64)
        for i in range(N):
            k = np.where(nx < M, key[s, np.arange(J) * M + np.minimum(nx, M - 1)], np.nan)
            best = min((kj, j) for j, kj in enumerate(k) if nx[j] < M)
            out[s, i] = best[1] * M + nx[best[1]]
            nx[best[1]] += 1
    return out


@pytest.mark.parametrize("source", ["random", "shipped"])
def test_priority_tables_give_back_the_rule_orders(source):
    if source == "shipped":
        g = np.load(PDR)
        t, p, J, M = g["t"], g["p"], 6, 6
    else:
        J, M = 7, 4
        d = ins.synthetic_instances(0, 12, J, M, 2, seed=5)
        t, p = d["t"], d["p"]
    for name in rules.OP_RULES:
        key, mach = rules.priority_table(name, "SEC", t, p, J, M)
        assert key.dtype == np.float64 and mach.dtype == np.int32 and key.shape == mach.shape == t.shape[:2]
        np.testing.assert_array_equal(_merge_by_key(key, J, M), rules.op_rule(name, t, p, J, M), err_msg=name)
        np.testing.assert_array_equal(mach, rules.machine_rule("SEC", t, p))


def test_argument_errors_without_a_device():
    lib = libm.lib()
    P = C.c_void_p(0x10000)
    for base in (0, 1, 2):
        assert lib.mtfjsp_complete(None, P, 4, P, 1, base, P, P, 0, 0, None, None, None, None, None) == E_ARG
        assert b"mtfjsp_complete" in lib.mtfjsp_last_error()


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _make(J, M, E, left_shift, d, w, mask_mode, B_=B):
    env = envm.BatchedMTFJSPEnv(B_, J, M, E, left_shift=left_shift, obs_dtype=torch.float32, mask_mode=mask_mode)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    env.obs()
    return env


def _data(J, M, E, seed, B_=B):
    return ins.synthetic_instances(0, B_, J, M, E, seed=seed), ins.random_weights(0, B_, seed=seed)


def _priority(d, J, M, seed):
    """A random priority table with a few ties, and SPT machines."""
    rng = np.random.default_rng(seed)
    key = rng.integers(0, 6, size=d["t"].shape[:2]).astype(np.float64) * 0.5
    key[rng.random(key.shape) < 0.1] = np.inf
    return key, rules.machine_rule("SPT", d["t"], d["p"]).astype(np.int32)


def _composed(env, left_shift, src, acts, base, key, mach, seed, mask_mode):
    """What complete must return: gather_from copies of env's envs src, stepped with the forced actions acts [T,R,2],
    then with policy_random(seed, 0, mask_mode) or the priority choice until done."""
    R = src.shape[0]
    N, J, M = env.N, env.J, env.M
    cp = envm.BatchedMTFJSPEnv(R, J, M, env.E, left_shift=left_shift, obs_dtype=torch.float32)
    cp.gather_from(env, src)
    dev = cp.device
    tot = torch.zeros((R, 5), dtype=torch.float64, device=dev)
    first = torch.full((R,), -1, dtype=torch.int32, device=dev)
    T = 0 if acts is None else acts.shape[0]
    for s in range(T):
        cp.step(acts[s, :, 0].contiguous(), acts[s, :, 1].contiguous())
        tot += cp.reward5
        first = torch.where((first < 0) & (cp.invalid != 0), s, first)
    bact = torch.full((N, R, 2), -1, dtype=torch.int32, device=dev)
    srcn = src.long().cpu().numpy()
    active = (cp.export_state()["mach"] >= 0).sum(1) < N
    for i in range(N + 1):
        if not bool(active.any()):
            break
        assert i < N
        if base == "random":
            op, mc = cp.policy_random(seed, 0, mask_mode)
            op, mc = op.clone(), mc.clone()
        else:
            _, _, _, _, jm, cand = cp.obs(mask_mode)
            jm, cand = jm.cpu().numpy(), cand.cpu().numpy()
            open_ = jm == 0
            kk = np.where(open_, key[srcn[:, None], cand] + 0.0, np.inf)
            j = np.argmax(open_ & (kk == kk.min(1, keepdims=True)), axis=1)        # the lowest open job of the least key
            op = cand[np.arange(R), j].astype(np.int32)
            mc = mach[srcn, op].astype(np.int32)
            op, mc = torch.as_tensor(op, device=dev), torch.as_tensor(mc, device=dev)
        op = torch.where(active, op, -1).to(torch.int32)
        mc = torch.where(active, mc, -1).to(torch.int32)
        bact[i] = torch.where(active[:, None], torch.stack((op, mc), 1), bact[i])
        cp.step(op, mc)
        tot += torch.where(active[:, None], cp.reward5, 0.0)
        bad = active & (cp.invalid != 0)
        first = torch.where((first < 0) & bad, T + i, first)
        active &= ~bad & (cp.done == 0)
    out = cp.costs(), tot, first, bact
    cp.close()
    return out


def _check(env, left_shift, src, acts, base, key, mach, seed, mask_mode, where):
    kd = None if key is None else torch.as_tensor(key, device=env.device)
    md = None if mach is None else torch.as_tensor(mach, device=env.device)
    got = env.complete(src, acts, base=base, key=kd, mach=md, seed=seed, mask_mode=mask_mode)
    exp = _composed(env, left_shift, src, acts, base, key, mach, seed, mask_mode)
    for name, g, e in zip(("final4", "return5", "first_invalid", "base_actions"), got, exp):
        np.testing.assert_array_equal(g.cpu().numpy(), e.cpu().numpy(), err_msg="%s %s" % (where, name))
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_complete_equals_the_composition(size, left_shift):
    J, M, E = size
    N = J * M
    d, w = _data(J, M, E, 60 + J)
    key, mach = _priority(d, J, M, J)
    dev = torch.device("cuda", torch.cuda.current_device())
    src = torch.tensor([4, 0, 0, 3, 1, 2, 4], dtype=torch.int32, device=dev)   # duplicated, permuted
    for mask_mode in (envm.MASK_FINISHED, envm.MASK_ESA):
        env = _make(J, M, E, left_shift, d, w, mask_mode)
        done = 0
        for stop in sorted({0, 1, N // 2, N - 1}):
            while done < stop:
                env.random_step(seed=11)
                done += 1
            cand = env.candidate_ops()
            a = torch.stack((cand[:, 0], torch.zeros_like(cand[:, 0])), 1)              # job 0's op on machine 0
            b = torch.stack((cand[:, -1], torch.ones_like(cand[:, -1])), 1)
            for T in (0, 1, 3):
                acts = None
                if T:
                    seq = torch.stack([a, b, torch.full_like(a, -1)][:T])                 # [T,B,2]; the last is invalid
                    if T == 1:
                        seq = torch.stack((cand[:, J - 1], torch.full_like(cand[:, 0], M - 1)), 1)[None]
                    acts = seq.index_select(1, src.long())
                for base in ("random", "priority"):
                    _check(env, left_shift, src, acts, base, key if base == "priority" else None, mach if base == "priority" else None,
                           5 + T, mask_mode, "mask %d step %d T %d %s" % (mask_mode, stop, T, base))
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"])
def test_complete_right_after_a_recorded_reset(fused, monkeypatch):
    monkeypatch.setenv("MTFJSP_FUSED_RESET", fused)
    J, M, E = 6, 6, 2
    d, w = _data(J, M, E, 23)
    env = _make(J, M, E, True, d, w, envm.MASK_ESA)
    key, mach = _priority(d, J, M, 1)
    for _ in range(9):
        env.random_step(seed=2)
    env.reset(w[::-1].copy())                                                   # recorded, performed by the call
    src = torch.tensor([1, 1, 0, 4, 3], dtype=torch.int32, device=env.device)
    _check(env, True, src, None, "random", None, None, 3, envm.MASK_ESA, "random")
    got = _check(env, True, src, None, "priority", key, mach, 0, envm.MASK_FINISHED, "priority")
    assert (got[2] == -1).all() and (got[3][:, :, 0] >= 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (30, 20, 5), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_complete_from_the_start_with_every_action_forced_equals_replay(size):
    J, M, E = size
    d, w = _data(J, M, E, 31)
    ref = _make(J, M, E, True, d, w, envm.MASK_ESA)
    acts = []
    for _ in range(J * M):
        ref.random_step(seed=4)
        acts.append(torch.stack((ref.op, ref.mach), 1).clone())
    acts = torch.stack(acts)
    env = _make(J, M, E, True, d, w, envm.MASK_ESA)
    src = torch.arange(B, dtype=torch.int32, device=env.device)
    f4, r5, fi, ba = env.complete(src, acts)
    for g, e in zip((f4, r5, fi), env.replay(acts)):
        np.testing.assert_array_equal(g.cpu().numpy(), e.cpu().numpy())
    assert (ba == -1).all() and (fi == -1).all()


def _state(env):
    st = env.export_state()
    sc = env.export_scaler()
    return [x.cpu().numpy() for x in list(st.values()) + list(sc.values()) + [env.costs(), env.candidate_ops()]]


@pytest.mark.gpu
def test_complete_leaves_the_env_untouched():
    from tests.test_env_peek import OUT
    J, M, E = 10, 10, 3
    N = J * M
    d, w = _data(J, M, E, 17)
    a = _make(J, M, E, True, d, w, envm.MASK_ESA)
    b = _make(J, M, E, True, d, w, envm.MASK_ESA)
    key, mach = _priority(d, J, M, 3)
    kd, md = torch.as_tensor(key, device=a.device), torch.as_tensor(mach, device=a.device)
    src = torch.tensor([1, 1, 0, 4, 2], dtype=torch.int32, device=a.device)
    for s in range(N):
        if s % 7 == 0:
            a.complete(src, base="random", seed=s)
            a.complete(src, base="priority", key=kd, mach=md, mask_mode=envm.MASK_FINISHED)
        a.policy_random(9, 0)
        op, mc = a.op.clone(), a.mach.clone()
        a.step_obs(op, mc)
        b.step_obs(op, mc)
        for x, y, n in zip([getattr(a, k) for k in OUT], [getattr(b, k) for k in OUT], OUT):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg="step %d %s" % (s, n))
    for x, y in zip(_state(a), _state(b)):
        np.testing.assert_array_equal(x, y)
    for mm in (envm.MASK_FINISHED, envm.MASK_ESA):
        for x, y in zip(a.obs(mm), b.obs(mm)):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy())
    f4, r5, fi, ba = a.complete(src, base="random")                              # every env is done: no base step
    assert (ba == -1).all() and (fi == -1).all() and (r5 == 0).all()
    np.testing.assert_array_equal(f4.cpu().numpy(), a.costs()[src.long()].cpu().numpy())


@pytest.mark.gpu
def test_errors_write_nothing_bad_sources_and_infeasible_key_machines():
    J, M, E = 6, 6, 2
    N = J * M
    d, w = _data(J, M, E, 29)
    lib = libm.lib()
    dev = torch.device("cuda", torch.cuda.current_device())
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    acts = torch.zeros((B, 1, 2), dtype=torch.int32, device=dev)
    src = torch.arange(B, dtype=torch.int32, device=dev)
    key = torch.zeros((B, N), dtype=torch.float64, device=dev)
    km = torch.zeros((B, N), dtype=torch.int32, device=dev)
    c4 = torch.full((B, 4), 7.0, dtype=torch.float64, device=dev)
    r5 = torch.full((B, 5), 7.0, dtype=torch.float64, device=dev)
    fi = torch.full((B,), 7, dtype=torch.int32, device=dev)
    ba = torch.full((B, N, 2), 7, dtype=torch.int32, device=dev)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h = env._h
    outs = (p(c4), p(r5), p(fi), p(ba), st)
    assert lib.mtfjsp_complete(h, p(src), B, p(acts), 1, 0, None, None, 0, 0, *outs) == E_STATE   # never reset
    env.scaler_init()
    env.reset(w)
    for args in [(None, p(src), B, p(acts), 1, 0, None, None), (h, None, B, p(acts), 1, 0, None, None),
                 (h, p(src), 0, p(acts), 1, 0, None, None), (h, p(src), B, p(acts), -1, 0, None, None),
                 (h, p(src), B, p(acts), N + 1, 0, None, None), (h, p(src), B, None, 1, 0, None, None),
                 (h, p(src), B, p(acts), 1, 2, None, None), (h, p(src), B, p(acts), 1, 1, None, p(km)),
                 (h, p(src), B, p(acts), 1, 1, p(key), None)]:
        assert lib.mtfjsp_complete(*args, 0, 0, *outs) == E_ARG
    assert lib.mtfjsp_complete(h, p(src), B, p(acts), 1, 0, None, None, 0, 2, *outs) == E_ARG      # bad mask_mode
    torch.cuda.synchronize()
    assert (c4 == 7.0).all() and (r5 == 7.0).all() and (fi == 7).all() and (ba == 7).all()
    bad = torch.tensor([0, -1, 2, B, 1 << 30], dtype=torch.int32, device=dev)
    got = env.complete(bad, base="random", seed=4)
    good = env.complete(torch.tensor([0, 0, 2, 0, 0], dtype=torch.int32, device=dev), base="random", seed=4)
    ok = torch.tensor([True, False, True, False, False], device=dev)
    for g, e in zip(got[:3], good[:3]):
        np.testing.assert_array_equal(g[ok].cpu().numpy(), e[ok].cpu().numpy())
        assert (g[~ok] == (-2 if g.dtype == torch.int32 else 0)).all()
    assert (got[3][:, ~ok] == -1).all()
    # an infeasible key_mach entry ends the run: FIFO order, op 7 on a machine it cannot use
    t = torch.as_tensor(d["t"], device=dev)
    kk = torch.arange(N, dtype=torch.float64, device=dev).expand(B, N).contiguous()
    mm = torch.as_tensor(rules.machine_rule("SPT", d["t"], d["p"]).astype(np.int32), device=dev)
    infeas = (t[:, 7] < 0).any(1)
    mm[:, 7] = torch.where(infeas, (t[:, 7] < 0).int().argmax(1), M).to(torch.int32)
    T = 2
    fa = torch.stack((torch.zeros(B, dtype=torch.int32, device=dev), mm[:, 0]), 1)[None].expand(T, B, 2).contiguous()
    fin = envm.MASK_FINISHED
    f4, r5_, fi_, ba_ = env.complete(src, fa, base="priority", key=kk, mach=mm, mask_mode=fin)  # step 1 repeats op 0
    assert (fi_ == 1).all()
    f4, r5_, fi_, ba_ = env.complete(src, fa[:1], base="priority", key=kk, mach=mm, mask_mode=fin)
    assert (fi_ == 1 + 6).all()                                                   # ops 1..6, then op 7 is invalid
    assert (ba_[6, :, 0] == 7).all() and (ba_[7:] == -1).all()


@pytest.mark.gpu
def test_priority_completions_reproduce_the_shipped_rule_rows():
    g = np.load(PDR)
    S = 100
    env = envm.BatchedMTFJSPEnv(S, 6, 6, 2, left_shift=False, obs_dtype=torch.float32, mask_mode=envm.MASK_FINISHED)
    env.load(g["t"], g["p"], g["transT"], g["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (S, 1)))
    src = torch.arange(S, dtype=torch.int32, device=env.device)
    for r, name in enumerate(str(x) for x in g["rule_names"]):
        o, m = name.split("+")
        key, mach = rules.priority_table(o, m, g["t"], g["p"], 6, 6)
        f4, _, fi, ba = env.complete(src, base="priority", key=torch.as_tensor(key, device=env.device),
                                     mach=torch.as_tensor(mach, device=env.device))
        np.testing.assert_array_equal(f4.cpu().numpy(), g["gold"][r], err_msg=name)
        np.testing.assert_array_equal(ba[:, :, 0].cpu().numpy().T, g["ops"][r].astype(np.int32), err_msg=name)
        assert (fi == -1).all()
