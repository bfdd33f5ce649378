"""mtfjsp_peek / BatchedMTFJSPEnv.peek: what a step would return for K (op, machine) pairs per env, without changing the
env.  Checked bit for bit against real steps (every env gathered into a copy per pair, then stepped) at specialised,
unspecialised and edge sizes, with and without left shift, at several points of an episode, for every candidate pair
and for invalid ones; the env is shown untouched by a twin fed the same actions; the lookahead rules built on it are
pinned to the reference's recorded runs (tests/golden/lookahead_golden.npz) and to an oracle restatement that replays
the prefix for every candidate.

Kernel mutations and the tests built to catch them: r_idle summed before the route follower's term is updated, or the
left-shift search skipped -> test_peek_equals_step (left_shift=True); the energy leaf of the peeked op not re-added
-> test_peek_equals_step, test_peek_reproduces_the_reference_it_temp, test_rules_equal_the_oracle_replay (GREEDY_R);
a global write left in the kernel -> test_peek_leaves_the_env_untouched."""
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
GOLD = os.path.join(os.path.dirname(__file__), "golden", "lookahead_golden.npz")
PDR = os.path.join(os.path.dirname(__file__), "golden", "pdr_golden.npz")
# specialised (J6M6, J10M10, J30M20: N > 128, the idle sum's chunk restart), unspecialised (J13M11), size edges
SIZES = [(6, 6, 2), (10, 10, 3), (30, 20, 5), (13, 11, 3), (70, 2, 1), (2, 64, 4)]
OUT = ["reward5", "scaled4", "done", "invalid", "task_fea", "mach_fea", "adj_w", "adj_src", "job_mask", "candidate"]


def _make(B, J, M, E, left_shift, d, w):
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    env.obs()
    return env


def _pairs(env, t):
    """[B,K] pairs: every (candidate op, machine) pair, then invalid ones -- an already-scheduled op, a later op of a job,
    an infeasible machine, out-of-range ops and machines."""
    B, J, M, N = env.B, env.J, env.M, env.N
    cand = env.candidate_ops()
    op = [cand.unsqueeze(2).expand(B, J, M).reshape(B, J * M)]
    mach = [torch.arange(M, dtype=torch.int32, device=env.device).repeat(J).expand(B, J * M)]
    sched = (env.export_state()["mach"] >= 0).to(torch.int32)
    done_op = torch.where(sched.any(dim=1), sched.argmax(dim=1).to(torch.int32), 0)           # a scheduled op (if any)
    later = torch.clamp(cand[:, 0] + 1, max=N - 1)                                             # job 0's next-but-one op
    c0 = cand[:, 0].long()
    tt = torch.as_tensor(t, device=env.device)[torch.arange(B, device=env.device), c0]        # [B,M]
    infeas = torch.where((tt < 0).any(dim=1), (tt < 0).to(torch.int32).argmax(dim=1), M).to(torch.int32)
    z = torch.zeros(B, dtype=torch.int32, device=env.device)
    extra = [(done_op, z), (later, z), (cand[:, 0], infeas), (z + N, z), (z - 1, z), (cand[:, 0], z + M),
             (cand[:, 0], z - 1)]
    op += [a[:, None] for a, _ in extra]
    mach += [m[:, None] for _, m in extra]
    return torch.cat(op, dim=1).contiguous(), torch.cat(mach, dim=1).contiguous()


def _check_against_steps(env, t, left_shift, where):
    op, mach = _pairs(env, t)
    B, K = op.shape
    r5, inv = env.peek(op, mach)
    cp = envm.BatchedMTFJSPEnv(B * K, env.J, env.M, env.E, left_shift=left_shift, obs_dtype=torch.float32)
    cp.gather_from(env, torch.arange(B, dtype=torch.int32, device=env.device).repeat_interleave(K))
    cp.step(op.reshape(-1).contiguous(), mach.reshape(-1).contiguous())
    np.testing.assert_array_equal(r5.reshape(-1, 5).cpu().numpy(), cp.reward5.cpu().numpy(), err_msg=where)
    np.testing.assert_array_equal(inv.reshape(-1).cpu().numpy(), cp.invalid.cpu().numpy(), err_msg=where)
    cp.close()
    return inv


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_peek_equals_step(size, left_shift):
    J, M, E = size
    N, B = J * M, 3
    d = ins.synthetic_instances(0, B, J, M, E, 500 + N)
    env = _make(B, J, M, E, left_shift, d, ins.random_weights(0, B, 5))
    at = sorted({0, 1, 3, N // 2, N - 1, N})
    s = 0
    for k in at:
        while s < k:
            env.random_step(seed=11, env_offset=0)
            s += 1
        inv = _check_against_steps(env, d["t"], left_shift, "J%dM%d ls=%d after %d steps" % (J, M, left_shift, k))
        if k < N:
            assert (inv[:, :J * M] == 0).any(dim=1).all()   # every live env has valid candidate pairs
        else:
            assert (inv == 1).all()                           # done envs: every pair invalid


def _snap(env):
    out = {n: getattr(env, n).cpu().numpy().copy() for n in OUT}
    out.update({"st_" + k: v.cpu().numpy() for k, v in env.export_state().items()})
    out.update({"sc_" + k: v.cpu().numpy() for k, v in env.export_scaler().items()})
    out["costs"] = env.costs().cpu().numpy()
    return out


def _same(a, b, where):
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg="%s: %s" % (where, k))


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (30, 20, 5), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_peek_leaves_the_env_untouched(size):
    """Twins fed the same actions (incremental observation on); one peeks every candidate pair between steps.  The
    state, scaler and costs, every output of the next fused step and of later back-to-back (overlapped) steps agree."""
    J, M, E = size
    N, B = J * M, 16
    d = ins.synthetic_instances(0, B, J, M, E, 700 + N)
    w = ins.random_weights(0, B, 6)
    a, b = _make(B, J, M, E, True, d, w), _make(B, J, M, E, True, d, w)
    for s in range(min(N, 24)):
        if s % 3 == 0:
            a.peek_candidates()
            a.peek_candidates(machines=torch.zeros((B, N), dtype=torch.int32, device=a.device))
        a.random_step(seed=3, env_offset=0)
        b.random_step(seed=3, env_offset=0)
        _same(_snap(a), _snap(b), "step %d" % s)
    a.peek_candidates()
    for _ in range(4):  # back to back: the later launches start overlapped where the size allows
        a.random_step(seed=4, env_offset=0)
        b.random_step(seed=4, env_offset=0)
    torch.cuda.synchronize()
    a.check_launch_overlap()
    _same(_snap(a), _snap(b), "overlapped")


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"])
def test_peek_after_a_recorded_reset(fused, monkeypatch):
    monkeypatch.setenv("MTFJSP_FUSED_RESET", fused)
    J, M, E, B = 6, 6, 2, 8
    d = ins.synthetic_instances(0, B, J, M, E, 901)
    w1, w2 = ins.random_weights(0, B, 1), ins.random_weights(0, B, 2)
    a = _make(B, J, M, E, True, d, w1)
    for _ in range(10):
        a.random_step(seed=5)
    a.reset(w2)                      # recorded: the peek must see the reset state
    fresh = _make(B, J, M, E, True, d, w2)
    ra, ia = a.peek_candidates()
    rf, if_ = fresh.peek_candidates()
    np.testing.assert_array_equal(ra.cpu().numpy(), rf.cpu().numpy())
    np.testing.assert_array_equal(ia.cpu().numpy(), if_.cpu().numpy())
    op = a.candidate_ops()[:, 2].contiguous()
    mach = ia[:, 2, :].to(torch.int32).argmin(dim=1).to(torch.int32)  # the first feasible machine of job 2's first op
    a.step(op, mach)
    fresh.step(op, mach)
    np.testing.assert_array_equal(a.reward5.cpu().numpy(), fresh.reward5.cpu().numpy())
    np.testing.assert_array_equal(a.export_state()["ft"].cpu().numpy(), fresh.export_state()["ft"].cpu().numpy())


@pytest.mark.gpu
def test_peek_errors_write_nothing():
    lib = libm.lib()
    J, M, E, B, K = 6, 6, 2, 4, 3
    d = ins.synthetic_instances(0, B, J, M, E, 903)
    env = envm.BatchedMTFJSPEnv(B, J, M, E)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    dev = env.device
    op = torch.zeros((B, K), dtype=torch.int32, device=dev)
    r5 = torch.full((B, K, 5), 7.25, dtype=torch.float64, device=dev)
    inv = torch.full((B, K), 9, dtype=torch.uint8, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.mtfjsp_peek(env._h, p(op), p(op), K, p(r5), p(inv), s) == E_STATE   # loaded, never reset
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 1))
    assert lib.mtfjsp_peek(None, p(op), p(op), K, p(r5), p(inv), s) == E_ARG
    assert lib.mtfjsp_peek(env._h, None, p(op), K, p(r5), p(inv), s) == E_ARG
    assert lib.mtfjsp_peek(env._h, p(op), None, K, p(r5), p(inv), s) == E_ARG
    assert lib.mtfjsp_peek(env._h, p(op), p(op), 0, p(r5), p(inv), s) == E_ARG
    torch.cuda.synchronize()
    assert (r5 == 7.25).all() and (inv == 9).all()
    # NULL outputs are allowed, each on its own
    assert lib.mtfjsp_peek(env._h, p(op), p(op), K, None, p(inv), s) == 0
    assert lib.mtfjsp_peek(env._h, p(op), p(op), K, p(r5), None, s) == 0
    torch.cuda.synchronize()
    assert (inv <= 1).all() and not (r5 == 7.25).any()


# ---- rules --------------------------------------------------------------------------------------------------------
def _gold_env(g, runs, J, M):
    t = np.stack([(g["t"] if J == 6 else g["t10"])[g["run_inst"][r]] for r in runs])
    p = np.stack([(g["p"] if J == 6 else g["p10"])[g["run_inst"][r]] for r in runs])
    tt = np.stack([(g["transT"] if J == 6 else g["transT10"])[g["run_inst"][r]] for r in runs])
    e = np.stack([(g["edge"] if J == 6 else g["edge10"])[g["run_inst"][r]] for r in runs])
    B = len(runs)
    env = envm.BatchedMTFJSPEnv(B, J, M, 2, left_shift=False)
    env.load(t, p, tt, e)
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (B, 1)))
    return env


@pytest.mark.gpu
def test_peek_reproduces_the_reference_it_temp():
    """Teacher-forced along every recorded run: peek_candidates(machines=machine list) gives every recorded it_temp bit
    for bit, and the reference's choice is in the device rule's arg-max set."""
    g = np.load(GOLD)
    for J, M in ((6, 6), (10, 10)):
        runs = [r for r in range(len(g["run_J"])) if g["run_J"][r] == J]
        env = _gold_env(g, runs, J, M)
        N, B = J * M, len(runs)
        ml = torch.as_tensor(g["mlist"][runs][:, :N].astype(np.int32), device=env.device)
        nx = np.zeros((B, J), dtype=np.int64)
        for s in range(N):
            r5, inv = env.peek_candidates(machines=ml)
            it, inv = r5[..., 2].cpu().numpy(), inv.cpu().numpy()
            ops = np.zeros(B, dtype=np.int32)
            for i, r in enumerate(runs):
                jobs = g["cand"][r, s][g["cand"][r, s] >= 0]
                np.testing.assert_array_equal(it[i, jobs], g["it"][r, s, :len(jobs)], err_msg="run %d step %d" % (r, s))
                assert (inv[i, jobs] == 0).all() and inv[i].sum() == J - len(jobs)
                best = it[i, jobs].max() if g["run_type"][r] == "min" else it[i, jobs].min()
                ch = int(g["chosen"][r, s])
                assert it[i, ch] == best, (r, s)
                ops[i] = ch * M + nx[i, ch]
                nx[i, ch] += 1
            opd = torch.as_tensor(ops, device=env.device)
            env.step(opd, torch.gather(ml, 1, opd.long()[:, None])[:, 0].contiguous())
        assert env.done.cpu().numpy().all()
        fin = env.costs().cpu().numpy()
        np.testing.assert_array_equal(fin, g["final4"][runs])


def _oracle_rollout(d, J, M, E, rule, mlist):
    """The rule by replay, on the oracle: per decision, one env per candidate pair replays the chosen prefix and steps
    its pair; lowest index among ties.  Returns actions [N,B,2] and final costs [B,4]."""
    from oracle.mtfjsp_oracle import OracleEnv

    B, N = d["t"].shape[0], J * M
    K = J * M if rule == "GREEDY_R" else J
    rep = lambda x: np.repeat(np.asarray(x), K, axis=0)
    env = OracleEnv(B * K, J, M, E, left_shift=False)
    env.load(rep(d["t"]), rep(d["p"]), rep(d["transT"]), rep(d["edge"]))
    acts = np.zeros((N, B, 2), dtype=np.int32)
    nx = np.zeros((B, J), dtype=np.int64)
    for s in range(N):
        env.scaler_init()
        env.reset(np.tile([0.4, 0.4, 0.2], (B * K, 1)))
        for a in acts[:s]:
            env.step(rep(a[:, 0]), rep(a[:, 1]))
        cand = np.arange(J)[None] * M + np.minimum(nx, M - 1)                    # [B,J]
        if rule == "GREEDY_R":
            op, mach = np.repeat(cand, M, axis=1), np.tile(np.arange(M), (B, J))
        else:
            op, mach = cand, np.take_along_axis(mlist, cand, axis=1)
        r5, _, _, inv = env.step(op.reshape(-1), mach.reshape(-1))
        r5, inv = r5.reshape(B, K, 5), inv.reshape(B, K)
        for b in range(B):
            ok = inv[b] == 0
            if rule == "GREEDY_R":
                v = np.where(ok, r5[b, :, 0], -np.inf); k = int(np.flatnonzero(v == v.max())[0])
            elif rule.startswith("LWKR_IT"):
                v = np.where(ok, r5[b, :, 2], -np.inf); k = int(np.flatnonzero(v == v.max())[0])
            else:
                v = np.where(ok, r5[b, :, 2], np.inf); k = int(np.flatnonzero(v == v.min())[0])
            acts[s, b] = (op[b, k], mach[b, k])
            nx[b, op[b, k] // M] += 1
    fin = OracleEnv(B, J, M, E, left_shift=False)
    fin.load(d["t"], d["p"], d["transT"], d["edge"])
    fin.scaler_init()
    fin.reset(np.tile([0.4, 0.4, 0.2], (B, 1)))
    for a in acts:
        fin.step(a[:, 0], a[:, 1])
    return acts, fin.costs()


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["LWKR_IT+SPT", "LWKR_IT+SEC", "MWKR_IT+SPT", "MWKR_IT+SEC", "GREEDY_R"])
@pytest.mark.parametrize("size", [(6, 6, 2, 8), (10, 10, 2, 16)], ids=["J6M6_shipped8", "J10M10_device16"])
def test_rules_equal_the_oracle_replay(size, rule):
    J, M, E, B = size
    if J == 6:
        d = ins.load_instances(os.path.join(os.path.dirname(__file__), "golden", "shipped_test_Instance_J6M6E2_first8.pkl"))
    else:
        d = {k: v.cpu().numpy() for k, v in ins.device_instances(0, B, J, M, E, seed=31).items()}
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=False)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (B, 1)))
    mlist = None
    if rule == "GREEDY_R":
        acts = rules.greedy_reward_rollout(env)
    else:
        name, mrule = rule.split("+")
        mlist = rules.machine_rule(mrule, d["t"], d["p"]).astype(np.int32)
        acts = rules.lookahead_rollout(env, name, torch.as_tensor(mlist, device=env.device))
    assert env.done.cpu().numpy().all() and not env.invalid.cpu().numpy().any()
    ref_acts, ref_costs = _oracle_rollout(d, J, M, E, rule, mlist)
    np.testing.assert_array_equal(acts.cpu().numpy(), ref_acts)
    np.testing.assert_array_equal(env.costs().cpu().numpy(), ref_costs)


@pytest.mark.gpu
def test_evaluate_rules_with_the_new_rows_on_the_shipped_instances():
    g = np.load(PDR)
    base = rules.evaluate_rules(g["t"], g["p"], g["transT"], g["edge"], 6, 6, 2)
    out = rules.evaluate_rules(g["t"], g["p"], g["transT"], g["edge"], 6, 6, 2,
                               op_rules=rules.OP_RULES + rules.LOOKAHEAD_RULES, joint_rules=rules.JOINT_RULES)
    R = len(base["names"])
    assert out["names"][:R] == base["names"] == [str(x) for x in g["rule_names"]]
    assert out["names"][R:] == ["LWKR_IT+SPT", "LWKR_IT+SEC", "MWKR_IT+SPT", "MWKR_IT+SEC", "GREEDY_R"]
    np.testing.assert_array_equal(out["costs"][:R], g["gold"])
    assert np.isfinite(out["costs"][R:]).all() and (out["costs"][R:] > 0).all()
