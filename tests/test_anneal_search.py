"""search.anneal_search, mtfjsp_anneal_propose / mtfjsp_anneal_step and their numpy restatements.  On the CPU:
exp_neg_reference against np.exp and at its edges, anneal_propose_reference against a brute-force enumeration of the
neighbourhood (with a row that has no move) and a chi-square test of its uniformity, anneal_step_reference against a
direct statement of the rules on forged states, and the argument errors.  On the GPU: both kernels against the references
bit for bit, the whole search against a CPU restatement on the oracle, its invariants and its independence of seed
repetition, chunking, batch and row."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
evolve = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.evolve")
validate = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
from oracle.mtfjsp_oracle import OracleEnv  # noqa: E402

W = (0.4, 0.4, 0.2)
E_ARG = -1
SIZES = [(3, 4, 2), (6, 6, 2), (10, 10, 3), (13, 11, 3), (70, 2, 1), (2, 64, 64), (30, 20, 5)]


def _forged_rows(J, M, Q, seed, p_infeasible=0.3):
    """Q random valid sequences of one forged J x M table t [1,N,M] (some entries infeasible, every op with at least one
    feasible machine), [Q,N,2] int32, each entry on a feasible machine."""
    rng = np.random.default_rng(seed)
    N = J * M
    t = rng.integers(1, 20, size=(1, N, M)).astype(np.float64)
    t[rng.random((1, N, M)) < p_infeasible] = -1.0
    t[0, np.arange(N), rng.integers(0, M, size=N)] = 5.0
    rows = np.empty((Q, N, 2), dtype=np.int32)
    for q in range(Q):
        jobs = rng.permutation(np.repeat(np.arange(J), M))
        seen = np.zeros(J, dtype=np.int64)
        for n, j in enumerate(jobs):
            o = j * M + seen[j]
            seen[j] += 1
            rows[q, n] = (o, rng.choice(np.flatnonzero(t[0, o] >= 0)))
    return t, rows


def _brute_neighbourhood(t_s, row):
    """The module docstring's neighbourhood of one sequence stated by loops: reassignments, then insertions."""
    N, M = t_s.shape
    pos = np.empty(N, dtype=np.int64)
    pos[row[:, 0]] = np.arange(N)
    out = []
    for s in range(N):
        o, m = int(row[s, 0]), int(row[s, 1])
        out += [(REASSIGN, s, mm) for mm in range(M) if t_s[o, mm] >= 0 and mm != m]
    for s in range(N):
        o = int(row[s, 0])
        lo = pos[o - 1] if o % M > 0 else -1
        hi = pos[o + 1] if o % M < M - 1 else N
        out += [(INSERT, s, sp) for sp in range(N) if lo < sp < hi and sp not in (s, s - 1)]
    return out


REASSIGN, INSERT = search.REASSIGN, search.INSERT


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_exp_neg_reference_within_one_ulp_and_at_its_edges():
    x = np.concatenate((np.linspace(0.0, 745.0, 1_000_001), np.random.default_rng(3).random(200_000) * 745.0))
    got, exp = search.exp_neg_reference(x), np.exp(-x)
    assert (np.abs(got - exp) <= np.spacing(exp)).all()
    assert search.exp_neg_reference(0.0) == 1.0
    np.testing.assert_array_equal(search.exp_neg_reference([-0.0, -1e-300, -5.0, -np.inf]), 1.0)
    np.testing.assert_array_equal(search.exp_neg_reference([746.5, 1e4, np.inf]), 0.0)
    assert np.isnan(search.exp_neg_reference(np.nan))
    sub = search.exp_neg_reference(np.array([709.0, 720.0, 740.0, 744.0]))
    assert ((sub > 0) & (sub < np.finfo(np.float64).tiny))[1:].all()
    assert not (np.random.default_rng(0).random() < search.exp_neg_reference(np.nan))


@pytest.mark.parametrize("size", [(3, 4), (2, 64), (70, 2), (30, 20)], ids=lambda s: "J%dM%d" % s)
def test_propose_reference_equals_brute_force(size):
    J, M = size
    K = 2 if J * M > 200 else 5
    t, rows = _forged_rows(J, M, K, seed=J * 100 + M)
    for it in (0, 7):
        got = search.anneal_propose_reference(t, rows, 11, it)
        for q in range(K):
            nb = _brute_neighbourhood(t[0], rows[q])
            u0 = evolve._draws(11, (it << 32) | q, 3)[0]
            kind, s, arg = nb[min(int(u0 * len(nb)), len(nb) - 1)]
            assert tuple(got[q]) == (q, kind, s, arg), (q, it)


def test_propose_reference_without_moves():
    # J1: one job in machine order, one feasible machine per op -> no reassignment and no insertion
    M = 4
    t = -np.ones((2, M, M))
    t[:, np.arange(M), np.arange(M)] = 3.0
    row = np.stack((np.arange(M), np.arange(M)), 1).astype(np.int32)
    rows = np.stack([row] * 6)                                                 # S = 2, K = 3
    got = search.anneal_propose_reference(t, rows, 0, 4)
    np.testing.assert_array_equal(got, [[q, -1, 0, 0] for q in range(6)])


def test_propose_reference_is_uniform_over_the_neighbourhood():
    stats = pytest.importorskip("scipy.stats")
    t, rows = _forged_rows(2, 3, 1, seed=5, p_infeasible=0.0)
    K = 64
    nb = _brute_neighbourhood(t[0], rows[0])
    counts = np.zeros(len(nb))
    for it in range(60):
        got = search.anneal_propose_reference(t, np.repeat(rows, K, 0), 9, it)
        for q in range(K):
            counts[nb.index(tuple(int(x) for x in got[q, 1:]))] += 1
    assert stats.chisquare(counts).pvalue > 1e-3


def _brute_step(state, moves, finv, obj, f4, temp, seed, it, parity, M):
    """The rules of include/mtfjsp.h stated directly, chain by chain and pair by pair."""
    st = {k: np.array(v, copy=True) for k, v in state.items()}
    S, K = temp.shape
    N = st["cur"].shape[1]
    st["accepted"][:] = 0
    st["swapped"][:] = 0
    u = np.stack([evolve._draws(seed, (it << 32) | k, 3) for k in range(K)])

    def p_accept(x):  # min(1, e^-x), NaN for NaN
        return math.nan if math.isnan(x) else (1.0 if x <= 0 else float(search.exp_neg_reference(x)))

    for q in range(S * K):
        s, k = divmod(q, K)
        row, kind, ms, arg = (int(x) for x in moves[q])
        if row != q or kind not in (0, 1) or not 0 <= ms < N or finv[q] != -1 or math.isnan(obj[q]):
            continue
        o, mo = (int(x) for x in st["cur"][q, ms])
        if not 0 <= o < N or not ((0 <= arg < M and 0 <= mo < M) if kind == 0 else 0 <= arg < N):
            continue
        d, T = obj[q] - st["cur_obj"][q], temp[s, k]
        if d <= 0 or (T > 0 and u[k, 1] < p_accept(d / T)):
            one = torch.tensor([[0, kind, ms, arg]])
            st["cur"][q] = search.apply_moves(torch.as_tensor(st["cur"][q][:, None]), one)[:, 0].numpy()
            st["cur_obj"][q], st["cur_f4"][q], st["accepted"][q] = obj[q], f4[q], 1
    if parity in (0, 1):
        for s in range(S):
            for k in range(parity, K - 1, 2):
                a, b = s * K + k, s * K + k + 1
                d, Ta, Tb = st["cur_obj"][b] - st["cur_obj"][a], temp[s, k], temp[s, k + 1]
                with np.errstate(divide="ignore", invalid="ignore"):
                    beta = np.float64(1.0) / Ta - np.float64(1.0) / Tb if Ta > 0 else math.nan
                if d <= 0 or (Ta > 0 and u[k, 2] < p_accept(d * beta)):
                    for key in ("cur", "cur_obj", "cur_f4"):
                        st[key][a], st[key][b] = st[key][b].copy(), st[key][a].copy()
                    st["swapped"][a] = 1
    for s in range(S):
        cand = [(st["cur_obj"][s * K + k], k) for k in range(K)
                if not math.isnan(st["cur_obj"][s * K + k]) and st["cur_obj"][s * K + k] < st["best_obj"][s]]
        if cand:
            v, k = min(cand)
            st["best"][s], st["best_obj"][s], st["best_f4"][s] = st["cur"][s * K + k], v, st["cur_f4"][s * K + k]
    return st


def _forged_step(seed, K, S=3, J=2, M=3):
    """A state of S instances x K chains at J x M with small-integer objectives (ties), its proposals from the reference
    with some malformed, NaN or invalid, and a ladder with zeros, equal and misordered temperatures."""
    rng = np.random.default_rng(seed)
    N = J * M
    t, rows = _forged_rows(J, M, S * K, seed=seed + 50)
    t = np.repeat(t, S, 0)
    f4 = rng.integers(0, 5, size=(S, 4)).astype(np.float64)
    st = search.anneal_state(rows[::K].copy(), f4, W, K)
    st["cur"] = rows.copy()
    st["cur_obj"] = rng.integers(0, 6, size=S * K).astype(np.float64)
    st["cur_f4"] = rng.random((S * K, 4))
    st["best_obj"] = st["best_obj"] - rng.integers(-2, 3, size=S)
    moves = search.anneal_propose_reference(t, rows, seed, 3)
    Q = S * K
    obj = rng.integers(0, 6, size=Q).astype(np.float64)
    obj[rng.random(Q) < 0.1] = np.nan
    st["cur_obj"][rng.random(Q) < 0.05] = np.nan
    finv = np.full(Q, -1, dtype=np.int32)
    finv[rng.random(Q) < 0.1] = 2
    bad = rng.random(Q) < 0.15
    moves[bad, rng.integers(0, 4, size=Q)[bad]] = rng.choice([-1, 2, N, 99], size=int(bad.sum()))
    mf4 = rng.random((Q, 4))
    temp = rng.choice([0.0, 0.5, 1.0, 2.0, 8.0], size=(S, K))                 # zeros, equal and misordered rungs
    return st, moves.astype(np.int32), finv, obj, mf4, temp


@pytest.mark.parametrize("K", [1, 2, 5, 8])
def test_step_reference_equals_the_rules_on_forged_states(K):
    took_then_swapped = 0
    for seed in range(8):
        st, moves, finv, obj, mf4, temp = _forged_step(seed, K)
        for parity in (-1, 0, 1):
            got = search.anneal_step_reference(st, moves, finv, obj, mf4, temp, seed, 4, parity, 3)
            exp = _brute_step(st, moves, finv, obj, mf4, temp, seed, 4, parity, 3)
            for k in st:
                np.testing.assert_array_equal(got[k], exp[k], err_msg="seed %d parity %d %s" % (seed, parity, k))
            took_then_swapped += int((got["accepted"] & (got["swapped"] | np.roll(got["swapped"], 1))).sum())
            if parity < 0 or K == 1:
                assert not got["swapped"].any()
    if K > 1:
        assert took_then_swapped > 0


def test_step_reference_ties_nan_and_temperatures():
    st, moves, finv, obj, mf4, temp = _forged_step(1, 4, S=1)
    finv[:] = -1
    moves = search.anneal_propose_reference(np.repeat(_forged_rows(2, 3, 4, seed=51)[0], 1, 0), st["cur"], 1, 3)
    st["cur_obj"][:] = 5.0
    st["best_obj"][:] = 9.0
    obj[:] = [5.0, 7.0, np.nan, 4.0]                                           # tie accepted, uphill at T=0 rejected
    temp = np.zeros((1, 4))
    got = search.anneal_step_reference(st, moves, finv, obj, mf4, temp, 0, 0, -1, 3)
    np.testing.assert_array_equal(got["accepted"], [1, 0, 0, 1])
    assert got["best_obj"][0] == 4.0
    np.testing.assert_array_equal(got["best"][0], got["cur"][3])
    obj[:] = [2.0, 2.0, 2.0, 2.0]                                              # best ties go to the lowest k
    got = search.anneal_step_reference(st, moves, finv, obj, mf4, temp, 0, 0, -1, 3)
    np.testing.assert_array_equal(got["best"][0], got["cur"][0])
    np.testing.assert_array_equal(got["best_f4"][0], mf4[0])
    # equal temperatures always swap; a pair whose upper chain is better always swaps
    obj[:] = np.nan
    st["cur_obj"][:] = [1.0, 3.0, 3.0, 2.0]
    got = search.anneal_step_reference(st, moves, finv, obj, mf4, np.full((1, 4), 2.0), 0, 0, 0, 3)
    np.testing.assert_array_equal(got["swapped"], [1, 0, 1, 0])
    np.testing.assert_array_equal(got["cur_obj"], [3.0, 1.0, 2.0, 3.0])


def test_entry_point_argument_errors_name_the_entry_point():
    lib = libm.lib()
    v = C.c_void_p(16)  # never dereferenced: every argument error is found before any launch

    def propose(t=v, S=2, J=2, M=3, K=4, cur=v, it=0, moves=v):
        return lib.mtfjsp_anneal_propose(t, S, J, M, K, cur, 1, it, moves, None)

    bad = [{"t": None}, {"cur": None}, {"moves": None}, {"S": 0}, {"K": 0}, {"J": 0}, {"M": 1}, {"M": 65},
           {"J": 600, "M": 20}, {"it": -1}, {"S": 1 << 16, "K": 1 << 16}]
    for kw in bad:
        assert propose(**kw) == E_ARG, kw
        assert b"mtfjsp_anneal_propose" in lib.mtfjsp_last_error()

    def step(S=2, J=2, M=3, K=4, ptrs=(v,) * 5, it=0, state=(v,) * 8):
        return lib.mtfjsp_anneal_step(S, J, M, K, *ptrs, 1, it, 0, *state, None)

    bad = [{"S": 0}, {"K": 0}, {"J": 0}, {"M": 1}, {"M": 65}, {"J": 600, "M": 20}, {"it": -1},
           {"S": 1 << 16, "K": 1 << 16}]
    bad += [{"ptrs": tuple(None if j == i else v for j in range(5))} for i in range(5)]
    bad += [{"state": tuple(None if j == i else v for j in range(8))} for i in range(8)]
    for kw in bad:
        assert step(**kw) == E_ARG, kw
        assert b"mtfjsp_anneal_step" in lib.mtfjsp_last_error()


def _random_sequences(J, M, E, S, seed, left_shift=True, chains=1):
    """Instances and `chains` random-rollout sequences of each from the oracle: [N, S*chains, 2], rows s*chains + k."""
    d = ins.synthetic_instances(0, S, J, M, E, seed=seed)
    Q = S * chains
    ora = OracleEnv(Q, J, M, E, left_shift=left_shift)
    ora.load(*(np.repeat(d[k], chains, 0) for k in ("t", "p", "transT", "edge")))
    ora.scaler_init()
    ora.reset(np.tile(np.asarray(W), (Q, 1)))
    acts = ora.rollout_random(J * M, seed, record_actions=True)["actions"]
    return {k: np.asarray(v) for k, v in d.items()}, acts


def test_search_argument_errors():
    d, acts = _random_sequences(3, 4, 2, 2, seed=1)
    for kw in ({"ladder": [0.2, 0.1]}, {"ladder": [-0.1, 0.1]}, {"ladder": [0.1, np.inf]}, {"ladder": [0.1, np.nan]},
               {"ladder": []}, {"ladder": [[0.1, 0.2]]}, {"iterations": -1}, {"swap_every": -1},
               {"max_candidates": 0}):
        with pytest.raises(ValueError):
            search.anneal_search(d, acts, **kw)
    with pytest.raises(ValueError):
        search.anneal_search(d, acts[:, :1])
    with pytest.raises(ValueError):
        search.anneal_search(d, acts[:-1])
    for K, hi, lo in ((0, 0.1, 0.01), (3, 0.01, 0.1), (3, 0.1, 0.0)):
        with pytest.raises(ValueError):
            search.anneal_ladder(K, hi, lo)
    lad = search.anneal_ladder(5, 0.1, 1e-3)
    assert lad[0] == 1e-3 and lad[-1] == 0.1 and (np.diff(lad) > 0).all()
    np.testing.assert_array_equal(search.anneal_ladder(1, 0.3, 0.01), [0.3])


# ---------------------------------------------------------------------------------------------------------------- GPU
def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _assert_state(dev_st, ref_st, where):
    for k in ref_st:
        np.testing.assert_array_equal(dev_st[k].cpu().numpy(), ref_st[k], err_msg="%s %s" % (where, k))


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_propose_kernel_equals_reference(size):
    J, M, E = size
    N = J * M
    S, K = (2, 3) if N > 200 else (3, 16)
    d, acts = _random_sequences(J, M, E, S, seed=N, chains=K)
    dev = _dev()
    cur = torch.as_tensor(acts, device=dev, dtype=torch.int32).transpose(0, 1).contiguous()
    t = torch.as_tensor(d["t"], device=dev, dtype=torch.float64)
    rows = cur.cpu().numpy()
    for it in (0, 1, 5, 123456):
        got = search.anneal_propose(t, cur, 77, it).cpu().numpy()
        np.testing.assert_array_equal(got, search.anneal_propose_reference(d["t"], rows, 77, it), err_msg=str(it))
    assert (got[:, 1] >= 0).all()


@pytest.mark.gpu
def test_propose_kernel_on_rows_without_moves_and_broken_rows():
    M = 4
    t = -np.ones((2, M, M))
    t[:, np.arange(M), np.arange(M)] = 3.0
    row = np.stack((np.arange(M), np.arange(M)), 1)
    rows = np.stack([row] * 6).astype(np.int32)
    rows[4, 1, 0] = 0                                                          # a duplicated op
    rows[5, 2, 0] = 77                                                         # an op out of range
    got = search.anneal_propose(torch.as_tensor(t, device=_dev()), torch.as_tensor(rows, device=_dev()), 0, 4)
    np.testing.assert_array_equal(got.cpu().numpy(), [[q, -1, 0, 0] for q in range(6)])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 2, 5, 8])
def test_step_kernel_equals_reference_on_forged_states(K):
    dev = _dev()
    for seed in range(6):
        st, moves, finv, obj, mf4, temp = _forged_step(seed, K)
        for parity in (-1, 0, 1):
            ref = search.anneal_step_reference(st, moves, finv, obj, mf4, temp, seed, 4, parity, 3)
            ds = {k: torch.as_tensor(v, device=dev) for k, v in st.items()}
            search.anneal_step(ds, *(torch.as_tensor(a, device=dev) for a in (moves, finv, obj, mf4, temp)), seed, 4,
                               parity, 3)
            _assert_state(ds, ref, "seed %d parity %d" % (seed, parity))


def _fresh_env(d, S, J, M, E, left_shift=True):
    env = envm.BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=W, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(W), (S, 1)))
    return env


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2, 4, 16, 50), (30, 20, 5, 2, 8, 50)], ids=("J6M6E2", "J30M20E5"))
def test_step_kernel_equals_reference_over_chained_iterations(size):
    J, M, E, S, K, iters = size
    d, acts = _random_sequences(J, M, E, S, seed=J + 3)
    env = _fresh_env(d, S, J, M, E)
    dev = env.device
    start = torch.as_tensor(acts, device=dev, dtype=torch.int32)
    f4, _, _ = env.replay(start)
    ds = search.anneal_state(start.transpose(0, 1).contiguous(), f4, W, K)
    ref = {k: v.cpu().numpy() for k, v in ds.items()}
    lad = search.anneal_ladder(K, 0.05, 1e-3)
    temp = torch.as_tensor(lad, device=dev)[None, :] * ds["best_obj"][:, None]
    t = torch.as_tensor(d["t"], device=dev, dtype=torch.float64)
    src = torch.arange(S * K, dtype=torch.int32, device=dev) // K
    taken = swaps = 0
    for it in range(iters):
        moves = search.anneal_propose(t, ds["cur"], 3, it)
        mf4, _, fi = env.replay_moves(ds["cur"].transpose(0, 1), moves, src)
        assert (fi == -1).all()
        obj = validate._objective(mf4, W)
        par = search._swap_parity(it, 2)
        search.anneal_step(ds, moves, fi, obj, mf4, temp, 3, it, par, M)
        ref = search.anneal_step_reference(ref, moves.cpu().numpy(), fi.cpu().numpy(), obj.cpu().numpy(),
                                           mf4.cpu().numpy(), temp.cpu().numpy(), 3, it, par, M)
        _assert_state(ds, ref, "iteration %d" % it)
        taken += int(ref["accepted"].sum())
        swaps += int(ref["swapped"].sum())
    assert 0 < taken < iters * S * K and swaps > 0


def _oracle_costs(d, seqs, src, left_shift):
    """final4 of the sequences seqs [N,R,2], row r replayed on instance src[r], by the oracle."""
    N, R, _ = seqs.shape
    M = d["t"].shape[2]
    ora = OracleEnv(R, N // M, M, d["edge"].shape[1], left_shift=left_shift)
    ora.load(*(d[k][src] for k in ("t", "p", "transT", "edge")))
    ora.scaler_init()
    ora.reset(np.tile(np.asarray(W), (R, 1)))
    for n in range(N):
        _, _, _, inv = ora.step(np.ascontiguousarray(seqs[n, :, 0]), np.ascontiguousarray(seqs[n, :, 1]))
        assert not inv.any()
    return ora.costs()


def _cpu_search(d, acts, iterations, ladder, swap_every, seed, left_shift=True):
    """anneal_search restated on the CPU: the reference kernels, apply_moves and oracle replays."""
    S, N, M = d["t"].shape
    K = len(ladder)
    f4 = _oracle_costs(d, acts, np.arange(S), left_shift)
    st = search.anneal_state(np.ascontiguousarray(acts.transpose(1, 0, 2)).astype(np.int32), f4, W, K)
    temp = np.asarray(ladder)[None, :] * st["best_obj"][:, None]
    hist = [st["best_obj"].copy()]
    src = np.arange(S * K) // K
    for it in range(iterations):
        moves = search.anneal_propose_reference(d["t"], st["cur"], seed, it)
        ok = moves[:, 1] >= 0
        mf4 = np.zeros((S * K, 4))
        fi = np.full(S * K, -2, dtype=np.int32)
        nb = search.apply_moves(torch.as_tensor(st["cur"].transpose(1, 0, 2)), torch.as_tensor(moves[ok])).numpy()
        mf4[ok] = _oracle_costs(d, nb, src[ok], left_shift)
        fi[ok] = -1
        st = search.anneal_step_reference(st, moves, fi, validate._objective(mf4, W), mf4, temp, seed, it,
                                          search._swap_parity(it, swap_every), M)
        hist.append(st["best_obj"].copy())
    return st, np.stack(hist)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(3, 4, 2), (6, 6, 2)], ids=("J3M4E2", "J6M6E2"))
def test_search_equals_cpu_restatement(size):
    J, M, E = size
    d, acts = _random_sequences(J, M, E, 3, seed=J * 7)
    lad = search.anneal_ladder(6, 0.1, 1e-3)
    for swap_every in (1, 3):
        out = search.anneal_search(d, acts, iterations=20, ladder=lad, swap_every=swap_every, seed=4)
        st, hist = _cpu_search(d, acts, 20, lad, swap_every, 4)
        np.testing.assert_array_equal(out["best_history"], hist)
        np.testing.assert_array_equal(out["actions"], st["best"].transpose(1, 0, 2))
        np.testing.assert_array_equal(out["final4"], st["best_f4"])
        np.testing.assert_array_equal(out["objective"], st["best_obj"])
        np.testing.assert_array_equal(out["current"], st["cur_obj"].reshape(3, 6))


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (10, 10, 3)], ids=("J6M6E2", "J10M10E3"))
def test_invariants(size):
    J, M, E = size
    d, acts = _random_sequences(J, M, E, 4, seed=8)
    out = search.anneal_search(d, acts, iterations=40, ladder=search.anneal_ladder(8, 0.05, 1e-3), seed=1)
    bh = out["best_history"]
    assert bh.shape == (41, 4) and out["current"].shape == (4, 8)
    assert out["accept_rate"].shape == (8,) and out["swap_rate"].shape == (7,) and out["replays"] == 4 + 40 * 32
    assert (np.diff(bh, axis=0) <= 0).all()
    f4, _, _ = _fresh_env(d, 4, J, M, E).replay(torch.as_tensor(acts, device=_dev(), dtype=torch.int32))
    np.testing.assert_array_equal(bh[0], validate._objective(f4, W).cpu().numpy())
    np.testing.assert_array_equal(bh[-1], out["objective"])
    got, _, fi = _fresh_env(d, 4, J, M, E).replay(torch.as_tensor(out["actions"], device=_dev()))
    assert (fi == -1).all()
    np.testing.assert_array_equal(got.cpu().numpy(), out["final4"])
    np.testing.assert_array_equal(validate._objective(out["final4"], W), out["objective"])
    assert (out["current"] >= out["objective"][:, None]).all()
    assert ((out["accept_rate"] > 0) & (out["accept_rate"] <= 1)).all()
    assert out["accept_rate"][-1] >= out["accept_rate"][0]


@pytest.mark.gpu
def test_zero_ladder_without_exchange_never_goes_uphill():
    d, acts = _random_sequences(6, 6, 2, 3, seed=12)
    env = _fresh_env(d, 3, 6, 6, 2)
    dev = env.device
    K = 4
    start = torch.as_tensor(acts, device=dev, dtype=torch.int32)
    f4, _, _ = env.replay(start)
    ds = search.anneal_state(start.transpose(0, 1).contiguous(), f4, W, K)
    temp = torch.zeros((3, K), dtype=torch.float64, device=dev)
    t = torch.as_tensor(d["t"], device=dev, dtype=torch.float64)
    src = torch.arange(3 * K, dtype=torch.int32, device=dev) // K
    prev = ds["cur_obj"].clone()
    for it in range(60):
        moves = search.anneal_propose(t, ds["cur"], 0, it)
        mf4, _, fi = env.replay_moves(ds["cur"].transpose(0, 1), moves, src)
        search.anneal_step(ds, moves, fi, validate._objective(mf4, W), mf4, temp, 0, it,
                           search._swap_parity(it, 0), 6)
        assert (ds["cur_obj"] <= prev).all() and not ds["swapped"].any()
        prev = ds["cur_obj"].clone()
    out = search.anneal_search(d, acts, iterations=60, ladder=np.zeros(K), swap_every=0)
    np.testing.assert_array_equal(out["best_history"][-1], ds["cur_obj"].view(3, K).min(1).values.cpu().numpy())
    np.testing.assert_array_equal(out["current"], ds["cur_obj"].view(3, K).cpu().numpy())
    assert np.isnan(out["swap_rate"]).all()


@pytest.mark.gpu
def test_reproducible_and_independent_of_chunking_batch_and_row():
    d, acts = _random_sequences(6, 6, 2, 6, seed=31)
    kw = dict(iterations=30, ladder=search.anneal_ladder(6, 0.05, 1e-3), seed=9)
    a = search.anneal_search(d, acts, **kw)
    b = search.anneal_search(d, acts, **kw)
    c = search.anneal_search(d, acts, max_candidates=7, **kw)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        np.testing.assert_array_equal(a[k], c[k], err_msg=k)
    for pick in (np.array([4]), np.array([5, 4, 0]), np.array([1, 4, 2, 3])):
        e = search.anneal_search({k: v[pick] for k, v in d.items()}, acts[:, pick], **kw)
        for k in ("best_history", "objective", "current", "final4"):
            np.testing.assert_array_equal(e[k], a[k][..., pick] if k == "best_history" else a[k][pick], err_msg=k)
        np.testing.assert_array_equal(e["actions"], a["actions"][:, pick])
