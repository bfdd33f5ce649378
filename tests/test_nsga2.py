"""NSGA-II (evolve.py) and its two kernels: the numpy specification of the non-dominated sorting rank against a
brute-force longest chain, the variation operator's numpy specification against an independent validity check (CPU);
mtfjsp_pareto_rank and mtfjsp_offspring against their specifications bit for bit, children replaying validly, and
nsga2's determinism, independence of chunking and batch, and elitism (GPU)."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pareto = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.pareto")
evolve = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.evolve")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
_lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SIZES = [(6, 6, 2), (13, 11, 3), (70, 2, 1), (2, 64, 4), (30, 20, 5)]
IMAX = np.iinfo(np.int32).max


def _random_sets(seed, big=False):
    """CSR point sets that exercise the edge cases: empty segments, a single point, integer coordinates with many ties,
    exact duplicates, continuous points, NaN and +-inf, a lattice front with dominated copies; with big, segments of
    more than 1,024 points and one of more than 4,096."""
    rng = np.random.default_rng(seed)
    segs = [np.zeros((0, 3)), rng.uniform(1, 5, (1, 3)), rng.integers(0, 4, (60, 3)).astype(np.float64),
            np.zeros((0, 3)), rng.uniform(0, 1, (90, 3))]
    dup = rng.integers(0, 6, (40, 3)).astype(np.float64)
    segs.append(np.concatenate((dup, dup[::3], dup[:5])))
    bad = rng.integers(0, 5, (50, 3)).astype(np.float64)
    bad[rng.integers(0, 50, 8), rng.integers(0, 3, 8)] = np.nan
    bad[rng.integers(0, 50, 4), rng.integers(0, 3, 4)] = np.inf
    bad[rng.integers(0, 50, 4), rng.integers(0, 3, 4)] = -np.inf
    segs.append(bad)
    a = rng.integers(0, 20, (70, 2))
    fr = np.stack((a[:, 0], a[:, 1], 40 - a[:, 0] - a[:, 1]), 1).astype(np.float64)
    segs.append(np.concatenate((fr, fr[:30] + rng.integers(0, 2, (30, 3)))))
    segs.append(np.repeat(rng.integers(0, 3, (1, 3)).astype(np.float64), 7, axis=0))       # one point seven times
    if big:
        segs.append(rng.integers(0, 12, (4096, 3)).astype(np.float64))
        segs.append(rng.integers(0, 40, (4097, 3)).astype(np.float64))
        c = rng.uniform(0, 1, (1500, 2))
        segs.append(np.stack((c[:, 0], c[:, 1], 2.0 - c[:, 0] - c[:, 1] + rng.uniform(0, 0.3, 1500)), 1))
    obj = np.concatenate(segs)
    seg = np.concatenate(([0], np.cumsum([len(s) for s in segs]))).astype(np.int64)
    return obj, seg


def _rank_chain(obj, seg):
    """Rank as the longest chain of beating points, by memoised recursion over the definition."""
    rank = np.zeros(len(obj), dtype=np.int64)
    for s in range(len(seg) - 1):
        a, b = int(seg[s]), int(seg[s + 1])
        fin = [bool(np.isfinite(obj[p]).all()) for p in range(a, b)]

        def beats(q, p):
            if not (fin[q - a] and fin[p - a]):
                return False
            le = all(obj[q, d] <= obj[p, d] for d in range(3))
            eq = all(obj[q, d] == obj[p, d] for d in range(3))
            return le and (not eq or q < p)

        memo = {}

        def chain(p):
            if p not in memo:
                memo[p] = max([chain(q) + 1 for q in range(a, b) if beats(q, p)], default=0)
            return memo[p]

        for p in range(a, b):
            rank[p] = chain(p) if fin[p - a] else IMAX
    return rank


def _valid(t, seqs, inst):
    """Independent validity of [N,C,2] sequences on instances inst [C]: every op once, each job's ops in order, every
    machine feasible."""
    S, N, M = t.shape
    for c in range(seqs.shape[1]):
        op, m = seqs[:, c, 0].astype(np.int64), seqs[:, c, 1].astype(np.int64)
        if not np.array_equal(np.sort(op), np.arange(N)):
            return False
        pos = np.empty(N, dtype=np.int64)
        pos[op] = np.arange(N)
        if not (np.diff(pos.reshape(N // M, M), axis=1) > 0).all():
            return False
        if not ((m >= 0) & (m < M)).all() or not (t[inst[c], op, m] >= 0).all():
            return False
    return True


def _random_parents(t, P, rng):
    """P valid sequences per instance ([N, S*P, 2], column s*P + k), drawn independently of the operator."""
    S, N, M = t.shape
    out = np.empty((N, S * P, 2), dtype=np.int32)
    for s in range(S):
        for k in range(P):
            x = rng.permutation(np.repeat(np.arange(N // M), M))
            cnt = np.zeros(N // M, dtype=np.int64)
            for i, j in enumerate(x):
                o = j * M + cnt[j]
                cnt[j] += 1
                out[i, s * P + k] = (o, rng.choice(np.flatnonzero(t[s, o] >= 0)))
    return out


def _case(J, M, E, S=3, P=4, C=24, seed=0):
    t = np.asarray(ins.synthetic_instances(0, S, J, M, E, seed=seed + 5)["t"])
    rng = np.random.default_rng(seed)
    par = _random_parents(t, P, rng)
    inst = rng.integers(0, S, C)
    pair = inst[:, None] * P + rng.integers(0, P, (C, 2))                     # parents of the child's instance
    pair[::5, 0] = -1                                                        # every fifth child random
    return t, par, pair, inst


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_rank_reference_equals_longest_chain(seed):
    obj, seg = _random_sets(seed)
    ref = pareto.pareto_rank_reference(obj, seg)
    np.testing.assert_array_equal(ref, _rank_chain(obj, seg))
    assert ref.max() > 2 and (ref == IMAX).any()
    np.testing.assert_array_equal(ref == 0, pareto.pareto_filter_reference(obj, seg))
    big = pareto.pareto_rank_reference(np.zeros((4097, 3)), [0, 4097])
    assert (big == -2).all()


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_offspring_reference_children_are_valid(size):
    t, par, pair, inst = _case(*size)
    for p_swap, p_mach in ((0.0, 0.0), (1.0, 0.3), (0.5, 1.0)):
        kids = evolve.offspring_reference(t, par, pair, inst, seed=17, p_swap=p_swap, p_mach=p_mach)
        assert _valid(t, kids, inst)


def test_offspring_reference_identical_parents_and_machine_sources():
    t, par, pair, inst = _case(13, 11, 3, P=4, C=40, seed=3)
    same = np.stack((pair[:, 1], pair[:, 1]), 1)
    kids = evolve.offspring_reference(t, par, same, inst, seed=9)
    np.testing.assert_array_equal(kids, par[:, same[:, 0]])
    pair[:, 0] = np.where(pair[:, 0] < 0, pair[:, 1], pair[:, 0])
    kids = evolve.offspring_reference(t, par, pair, inst, seed=9, p_swap=1.0)
    N = t.shape[1]
    for c in range(pair.shape[0]):
        by_op = np.empty((2, N), dtype=np.int64)
        for r in range(2):
            by_op[r, par[:, pair[c, r], 0]] = par[:, pair[c, r], 1]
        m = np.empty(N, dtype=np.int64)
        m[kids[:, c, 0]] = kids[:, c, 1]
        assert ((m == by_op[0]) | (m == by_op[1])).all()
    # both parents' machines are used, and the children differ from both parents
    assert any((kids[:, c] != par[:, pair[c, 0]]).any() and (kids[:, c] != par[:, pair[c, 1]]).any()
               for c in range(pair.shape[0]))


def test_offspring_bad_parents_and_argument_errors():
    t, par, pair, inst = _case(6, 6, 2)
    pair[1] = (-2, 0)
    pair[2] = (0, par.shape[1])
    inst[3] = -1
    kids = evolve.offspring_reference(t, par, pair, inst, seed=1)
    assert (kids[:, 1:4] == -1).all() and (kids[:, 4:] >= 0).all()
    lib = _lib.lib()
    v = C.c_void_p(16)
    assert lib.mtfjsp_offspring(None, 1, 6, 6, v, 1, v, v, 1, 0, 0.0, 0.0, v, None) == -1
    assert lib.mtfjsp_offspring(v, 1, 6, 6, v, 1, v, v, -1, 0, 0.0, 0.0, v, None) == -1
    assert lib.mtfjsp_offspring(v, 1, 6, 65, v, 1, v, v, 1, 0, 0.0, 0.0, v, None) == -1
    assert lib.mtfjsp_offspring(v, 1, 600, 20, v, 1, v, v, 1, 0, 0.0, 0.0, v, None) == -1
    assert lib.mtfjsp_offspring(v, -1, 6, 6, v, 1, v, v, 1, 0, 0.0, 0.0, v, None) == -1
    assert lib.mtfjsp_offspring(v, 1, 6, 6, v, -1, v, v, 1, 0, 0.0, 0.0, v, None) == -1
    assert b"mtfjsp_offspring" in lib.mtfjsp_last_error()
    assert lib.mtfjsp_pareto_rank(None, v, 1, 1, v, None) == -1
    assert lib.mtfjsp_pareto_rank(v, v, -1, 1, v, None) == -1
    assert lib.mtfjsp_pareto_rank(v, v, 1, -1, v, None) == -1
    assert b"mtfjsp_pareto_rank" in lib.mtfjsp_last_error()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _replay(t_inst, seqs, src, left_shift):
    S, N, M = t_inst["t"].shape
    env = envm.BatchedMTFJSPEnv(S, N // M, M, t_inst["edge"].shape[1], left_shift=left_shift, obs_dtype=torch.float32)
    env.load(t_inst["t"], t_inst["p"], t_inst["transT"], t_inst["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (S, 1)))
    f4, _, fi = env.replay(torch.as_tensor(seqs, device=env.device), torch.as_tensor(src, device=env.device))
    out = f4.cpu().numpy(), fi.cpu().numpy()
    env.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1])
def test_rank_kernel_equals_reference(seed):
    obj, seg = _random_sets(seed, big=True)
    want = pareto.pareto_rank_reference(obj, seg)
    assert (want == -2).any()
    o, s = torch.as_tensor(obj, device="cuda"), torch.as_tensor(seg, device="cuda")
    for max_len in (None, 0, 100, 4096, 10000):     # below a segment's length: that segment is read from global memory
        np.testing.assert_array_equal(pareto.pareto_rank(o, s, max_len=max_len).cpu().numpy(), want)
    small = want != -2                                                      # the filter has no segment limit
    np.testing.assert_array_equal((pareto.pareto_rank(o, s).cpu().numpy() == 0)[small],
                                  pareto.pareto_filter(o, s).cpu().numpy()[small])
    assert pareto.pareto_rank(o[:0], torch.zeros(3, dtype=torch.int64, device="cuda")).numel() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_offspring_kernel_equals_reference_and_replays(size):
    J, M, E = size
    S = 3
    d = {k: np.asarray(v) for k, v in ins.synthetic_instances(0, S, J, M, E, seed=5).items()}
    t, par, pair, inst = _case(J, M, E, S=S, C=40)
    pair[7] = (-3, 0)                                                       # bad parent indices: -1 rows
    pair[8] = (1, par.shape[1])
    for seed, p_swap, p_mach in ((3, 0.0, 0.0), (4, 1.0, 0.2), (2 ** 63 + 5, 0.3, 1.0)):
        want = evolve.offspring_reference(t, par, pair, inst, seed=seed, p_swap=p_swap, p_mach=p_mach)
        got = evolve.offspring(t, torch.as_tensor(par, device="cuda"), pair, inst, seed=seed, p_swap=p_swap,
                               p_mach=p_mach).cpu().numpy()
        np.testing.assert_array_equal(got, want)
        assert (got[:, 7:9] == -1).all()
        ok = np.setdiff1d(np.arange(pair.shape[0]), [7, 8])
        for ls in (True, False):
            _, fi = _replay(d, got[:, ok], inst[ok].astype(np.int32), ls)
            assert (fi == -1).all()


def _shipped():
    return ins.load_instances(os.path.join(GOLD, "shipped_test_Instance_J6M6E2_first8.pkl"))


@pytest.mark.gpu
def test_nsga2_deterministic_and_independent_of_chunking_and_batch():
    d = {k: np.asarray(v) for k, v in _shipped().items()}
    kw = dict(pop=24, generations=5, seed=11)
    a = evolve.nsga2(d, **kw)
    b = evolve.nsga2(d, **kw)
    c = evolve.nsga2(d, max_candidates=64, **kw)
    e = evolve.nsga2(d, max_candidates=65536, **kw)
    for k in ("actions", "final4", "objectives", "rank", "ref", "hypervolume"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        np.testing.assert_array_equal(a[k], c[k], err_msg=k)
        np.testing.assert_array_equal(a[k], e[k], err_msg=k)
    assert a["replays"] == 8 * 24 * 6
    alone = evolve.nsga2({k: v[:1] for k, v in d.items()}, **kw)
    for k in ("final4", "objectives", "rank", "ref", "hypervolume"):
        np.testing.assert_array_equal(alone[k], a[k][:, :1] if k == "hypervolume" else a[k][:1], err_msg=k)
    np.testing.assert_array_equal(alone["actions"], a["actions"][:, :1])
    # row 3 keeps its instance while every other row holds another one: row 3's result is unchanged
    perm = np.array([5, 7, 6, 3, 1, 0, 2, 4])
    mixed = evolve.nsga2({k: v[perm] for k, v in d.items()}, **kw)
    for k in ("final4", "objectives", "rank", "ref"):
        np.testing.assert_array_equal(mixed[k][3], a[k][3], err_msg=k)
    np.testing.assert_array_equal(mixed["hypervolume"][:, 3], a["hypervolume"][:, 3])
    np.testing.assert_array_equal(mixed["actions"][:, 3], a["actions"][:, 3])
    # every member replays to its recorded costs
    N = d["t"].shape[1]
    f4, fi = _replay(d, a["actions"].reshape(N, -1, 2), np.repeat(np.arange(8, dtype=np.int32), 24), True)
    assert (fi == -1).all()
    np.testing.assert_array_equal(f4, a["final4"].reshape(-1, 4))


@pytest.mark.gpu
def test_nsga2_elitism_from_a_start_set():
    d = {k: np.asarray(v) for k, v in _shipped().items()}
    S, N, M = d["t"].shape
    rng = np.random.default_rng(4)
    start = _random_parents(d["t"], 6, rng).reshape(N, S, 6, 2).transpose(0, 2, 1, 3)   # [N,K,S,2]
    out = evolve.nsga2(d, start, pop=512, generations=8, seed=2)
    assert (out["rank"] < 512).all()
    front_sizes = (out["rank"] == 0).sum(1)
    assert (front_sizes < 512).all()                                           # front 0 was never truncated
    h = out["hypervolume"]
    assert h.shape == (9, S)
    # the FP64 volume of a region that only grows may move by rounding when a point is replaced by one an ulp away
    assert (np.diff(h, axis=0) >= -1e-12 * h[1:]).all()
    assert (h[-1] > h[0]).all()
    f4, fi = _replay(d, start.reshape(N, -1, 2), np.tile(np.arange(S, dtype=np.int32), 6), True)
    assert (fi == -1).all()
    so = pareto.objectives(f4).reshape(6, S, 3)
    for s in range(S):
        fr = out["objectives"][s][out["rank"][s] == 0]
        assert pareto.pareto_filter_reference(fr, [0, len(fr)]).all()
        for p in so[:, s]:
            assert (fr <= p).all(axis=1).any()
    bad = start.copy()
    bad[1, 0, 0] = bad[0, 0, 0]
    with pytest.raises(ValueError):
        evolve.nsga2(d, bad, pop=8, generations=1)
