"""pareto.py: the numpy specifications of the dominance filter and of the exact hypervolume against independent brute
forces, the crowding-distance cut and the weighted-sum bits of `objectives` (CPU); the two kernels of mtfjsp_pareto.cu
against the specifications bit for bit, and the fronts of sampled validation (GPU)."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pareto = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.pareto")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
_lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _random_sets(seed, big=False):
    """CSR point sets that exercise the edge cases: empty segments, a single point, integer coordinates with many ties,
    exact duplicates, continuous points, NaN and inf; with big, segments of more than one tile."""
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
    # a front plus dominated points: x + y + z = const on a lattice, then shifted copies
    a = rng.integers(0, 20, (70, 2))
    fr = np.stack((a[:, 0], a[:, 1], 40 - a[:, 0] - a[:, 1]), 1).astype(np.float64)
    segs.append(np.concatenate((fr, fr[:30] + rng.integers(0, 2, (30, 3)))))
    if big:
        segs.append(rng.integers(0, 40, (5000, 3)).astype(np.float64))
        c = rng.uniform(0, 1, (3000, 2))
        segs.append(np.stack((c[:, 0], c[:, 1], 2.0 - c[:, 0] - c[:, 1]), 1))
        segs.append(np.concatenate((np.zeros((0, 3)), rng.uniform(0, 1, (700, 3)))))
    obj = np.concatenate(segs)
    seg = np.concatenate(([0], np.cumsum([len(s) for s in segs]))).astype(np.int64)
    return obj, seg


def _filter_loop(obj, seg):
    keep = np.zeros(len(obj), dtype=bool)
    for s in range(len(seg) - 1):
        for p in range(seg[s], seg[s + 1]):
            if not np.isfinite(obj[p]).all():
                continue
            ok = True
            for q in range(seg[s], seg[s + 1]):
                if q == p or not np.isfinite(obj[q]).all():
                    continue
                le = all(obj[q, d] <= obj[p, d] for d in range(3))
                lt = any(obj[q, d] < obj[p, d] for d in range(3))
                eq = all(obj[q, d] == obj[p, d] for d in range(3))
                if (le and lt) or (eq and q < p):
                    ok = False
                    break
            keep[p] = ok
    return keep


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_filter_reference_equals_a_plain_loop(seed):
    obj, seg = _random_sets(seed)
    ref = pareto.pareto_filter_reference(obj, seg)
    np.testing.assert_array_equal(ref, _filter_loop(obj, seg))
    assert ref.any() and not ref.all()


def _hv_grid(u):
    """Exact volume of the union of boxes [u_i, 1]^3 by coordinate compression: every cell of the grid of the points'
    coordinates and 1.0 is inside the union iff some point is <= its lower corner."""
    if len(u) == 0:
        return 0.0
    axes = [np.unique(np.append(u[:, d], 1.0)) for d in range(3)]
    lo = np.meshgrid(*[a[:-1] for a in axes], indexing="ij")
    width = np.meshgrid(*[np.diff(a) for a in axes], indexing="ij")
    cov = np.zeros(lo[0].shape, dtype=bool)
    for p in u:
        cov |= (p[0] <= lo[0]) & (p[1] <= lo[1]) & (p[2] <= lo[2])
    return float((width[0] * width[1] * width[2] * cov).sum())


@pytest.mark.parametrize("seed", range(6))
def test_hypervolume_reference_equals_grid_enumeration(seed):
    rng = np.random.default_rng(100 + seed)
    segs, refs, want = [], [], []
    for n in (0, 1, 2, 5, 17, 40):
        v = rng.uniform(0.5, 10, (n, 3)) if seed % 2 else rng.integers(1, 8, (n, 3)).astype(np.float64)
        r = np.array([9.0, 11.0, 10.0])
        if n > 3:
            v[0] = r + 1.0           # outside the box: takes no part
            v[1, 2] = np.nan         # non-finite: takes no part
        u = v / r
        u = u[np.isfinite(u).all(1) & (u < 1).all(1)]
        segs.append(v)
        refs.append(r)
        want.append(_hv_grid(u))
    obj = np.concatenate(segs)
    seg = np.concatenate(([0], np.cumsum([len(s) for s in segs]))).astype(np.int64)
    got = pareto.hypervolume3_reference(obj, seg, np.array(refs))
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert got[0] == 0.0


def test_hypervolume_reference_edges():
    one = pareto.hypervolume3_reference([[1.0, 2.0, 3.0]], [0, 1], [[4.0, 4.0, 4.0]])
    assert one[0] == (1 - 0.25) * (1 - 0.5) * (1 - 0.75)
    out = pareto.hypervolume3_reference(np.zeros((4098, 3)), [0, 4097, 4097, 4098, 4098],
                                        [[1.0, 1.0, 1.0], [1.0, 1.0, 1.0], [1.0, np.inf, 1.0], [1.0, 0.0, 1.0]])
    assert np.isnan(out[0]) and out[1] == 0.0 and np.isnan(out[2]) and np.isnan(out[3])


def test_crowding_truncation_keeps_the_extremes_and_is_deterministic():
    rng = np.random.default_rng(7)
    # two groups of points on a front, with tied coordinates and a tied crowding distance
    a = rng.integers(0, 12, (40, 2))
    g0 = np.stack((a[:, 0], a[:, 1], 30 - a[:, 0] - a[:, 1]), 1).astype(np.float64)
    g1 = np.array([[0, 4, 4], [1, 3, 4], [2, 2, 4], [3, 1, 4], [4, 0, 4]], dtype=np.float64)  # tt constant
    obj = torch.as_tensor(np.concatenate((g0, g1)))
    inst = torch.as_tensor(np.r_[np.zeros(40), np.ones(5)].astype(np.int64))
    cd = pareto.crowding_distance(obj, inst, 2).numpy()
    # the equal spacing of g1: interior points have crowding 2/4 (mk) + 2/4 (ec) + 0 (tt range 0)
    np.testing.assert_array_equal(cd[40:], [np.inf, 1.0, 1.0, 1.0, np.inf])
    for cap in (6, 9, 20):
        keep = pareto.crowding_truncate(obj, inst, 2, cap).numpy()
        assert keep[:40].sum() == cap and keep[40:].sum() == min(5, cap)
        for d in range(3):  # the lowest-index minimum and maximum of every objective are boundary points: kept
            v = g0[:, d]
            assert keep[np.flatnonzero(v == v.min())[0]] and keep[np.flatnonzero(v == v.max())[-1]]
        np.testing.assert_array_equal(keep, pareto.crowding_truncate(obj, inst, 2, cap).numpy())
    keep = pareto.crowding_truncate(obj, inst, 2, 3).numpy()
    np.testing.assert_array_equal(keep[40:], [True, True, False, False, True])  # the tie at 1.0 goes to the lower index


def test_objectives_keep_the_weighted_sum_bits():
    rng = np.random.default_rng(3)
    f4 = rng.uniform(0, 500, (7, 33, 4))
    f4[..., 0] = np.round(f4[..., 0])
    for w in ((0.4, 0.4, 0.2), (0.25, 0.5, 0.25), (1.0, 0.0, 0.0), (0.1, 0.7, 0.2)):
        o = pareto.objectives(f4)
        np.testing.assert_array_equal(w[0] * o[..., 0] + w[1] * o[..., 1] + w[2] * o[..., 2], val._objective(f4, w))
        ot = pareto.objectives(torch.as_tensor(f4))
        np.testing.assert_array_equal(ot.numpy(), o)


def test_argument_errors_return_codes():
    lib = _lib.lib()
    p = C.c_void_p(16)
    assert lib.mtfjsp_pareto_filter(None, p, 1, 1, p, None) == -1
    assert lib.mtfjsp_pareto_filter(p, None, 1, 1, p, None) == -1
    assert lib.mtfjsp_pareto_filter(p, p, 1, 1, None, None) == -1
    assert lib.mtfjsp_pareto_filter(p, p, -1, 1, p, None) == -1
    assert lib.mtfjsp_pareto_filter(p, p, 1, -1, p, None) == -1
    assert lib.mtfjsp_hypervolume3(None, p, 1, p, p, None) == -1
    assert lib.mtfjsp_hypervolume3(p, None, 1, p, p, None) == -1
    assert lib.mtfjsp_hypervolume3(p, p, 1, None, p, None) == -1
    assert lib.mtfjsp_hypervolume3(p, p, 1, p, None, None) == -1
    assert lib.mtfjsp_hypervolume3(p, p, -1, p, p, None) == -1


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_filter_kernel_equals_reference(seed):
    obj, seg = _random_sets(seed, big=True)
    want = pareto.pareto_filter_reference(obj, seg)
    o, s = torch.as_tensor(obj, device="cuda"), torch.as_tensor(seg, device="cuda")
    np.testing.assert_array_equal(pareto.pareto_filter(o, s).cpu().numpy(), want)
    for max_len in (0, 1, 300):  # a grid smaller than the longest segment needs: the blocks stride over it
        np.testing.assert_array_equal(pareto.pareto_filter(o, s, max_len=max_len).cpu().numpy(), want)
    # no segments, and every point in empty segments
    assert pareto.pareto_filter(o[:0], torch.zeros(1, dtype=torch.int64, device="cuda")).numel() == 0
    z = torch.zeros(4, dtype=torch.int64, device="cuda")
    assert not pareto.pareto_filter(o[:0], z).any()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1])
def test_hypervolume_kernel_equals_reference(seed):
    rng = np.random.default_rng(50 + seed)
    segs, refs = [], []
    for n in (0, 1, 3, 40, 257, 1000, 4096, 4097, 5):
        if n % 2:
            v = rng.integers(1, 30, (n, 3)).astype(np.float64)
        else:
            c = rng.uniform(0.1, 1.0, (n, 2))
            v = np.stack((c[:, 0], c[:, 1], 2.5 - c[:, 0] - c[:, 1] + rng.uniform(0, 0.2, n)), 1) * 37.0
        if n > 10:
            v[rng.integers(0, n, 3), rng.integers(0, 3, 3)] = np.nan
            v[rng.integers(0, n, 3)] = 1e9
        segs.append(v)
        refs.append(1.1 * np.nanmax(np.where(v >= 1e9, np.nan, v), axis=0) if n > 1 else np.array([40.0, 40.0, 90.0]))
    refs[-1] = np.array([40.0, -1.0, 90.0])          # a bad reference point
    obj = np.concatenate(segs)
    seg = np.concatenate(([0], np.cumsum([len(s) for s in segs]))).astype(np.int64)
    ref = np.array(refs)
    want = pareto.hypervolume3_reference(obj, seg, ref)
    got = pareto.hypervolume(torch.as_tensor(obj, device="cuda"), torch.as_tensor(seg, device="cuda"), ref).cpu().numpy()
    np.testing.assert_array_equal(got.view(np.int64), want.view(np.int64))
    assert got[0] == 0.0 and np.isnan(got[7]) and np.isnan(got[8]) and np.isfinite(got[:7]).all() and (got[1:7] > 0).all()
    # the volume of a set is the volume of its front
    keep = pareto.pareto_filter_reference(obj, seg)
    cnt = np.array([keep[seg[s]:seg[s + 1]].sum() for s in range(len(seg) - 1)])
    fr = pareto.hypervolume(torch.as_tensor(obj[keep], device="cuda"), np.r_[0, np.cumsum(cnt)], ref).cpu().numpy()
    np.testing.assert_allclose(fr[:7], got[:7], rtol=1e-12)


@pytest.mark.gpu
def test_front_of_sampled_validation_holds_the_best_objective():
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k][:24] for k in ("t", "p", "transT", "edge")}
    op_sd, mch_sd = val.load_actor_state_dicts(os.path.join(GOLD, "policy_golden.npz"), "iotj")
    ja = enc.JobActor(op_sd, 6, 6, precision="tf32")
    ma = enc.MachineActor(mch_sd, 6, precision="tf32")
    sp = val.sampled_validate(ja, ma, inst, 64, seed=3)
    fr = pareto.front(sp["final4"])
    obj = pareto.objectives(sp["final4"])                                   # [K,S,3]
    w = np.array([0.4, 0.4, 0.2])
    for s, idx in enumerate(fr):
        assert len(idx) >= 1 and (np.diff(idx) > 0).all()
        assert min(val._objective(sp["final4"][idx, s], (0.4, 0.4, 0.2))) == sp["best_objective"][s]
        want = np.flatnonzero(pareto.pareto_filter_reference(obj[:, s], [0, 64]))
        np.testing.assert_array_equal(idx, want)
        o = obj[idx, s]
        assert (w[0] * o[:, 0] + w[1] * o[:, 1] + w[2] * o[:, 2]).min() == sp["best_objective"][s]
    tab = pareto.hypervolume_table({"sampled": sp["final4"], "best": sp["best_final4"]})
    assert (tab["hypervolume"]["sampled"] >= tab["hypervolume"]["best"]).all()
    np.testing.assert_array_equal(tab["union"], tab["hypervolume"]["sampled"])
