"""search.pareto_local_search on mtfjsp_replay and mtfjsp_pareto_filter (GPU): archive members replay plainly, are
mutually non-dominated and weakly dominate the start set; the hypervolume never falls (beyond rounding); at natural termination no
neighbour of any member survives an archive-first filter; determinism, independence of chunking and batch; truncation."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
pareto = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.pareto")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
from oracle.mtfjsp_oracle import OracleEnv  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
KEYS = ("actions", "final4", "objectives", "count", "explored", "ref", "hypervolume", "truncated")


def _start(J, M, E, S, K, seed, d=None):
    """K random valid sequences per instance of S synthetic instances (or of the instances d): [N,K,S,2]."""
    if d is None:
        d = {k: np.asarray(v) for k, v in ins.synthetic_instances(0, S, J, M, E, seed=seed).items()}
    rep = {k: np.tile(v, (K,) + (1,) * (v.ndim - 1)) for k, v in d.items()}
    ora = OracleEnv(K * S, J, M, E, left_shift=True)
    ora.load(rep["t"], rep["p"], rep["transT"], rep["edge"])
    ora.scaler_init()
    ora.reset(np.tile([0.4, 0.4, 0.2], (K * S, 1)))
    acts = ora.rollout_random(J * M, seed, record_actions=True)["actions"]
    return d, acts.reshape(J * M, K, S, 2)


def _replay_plain(inst, seqs, src):
    S, N, M = inst["t"].shape
    env = envm.BatchedMTFJSPEnv(S, N // M, M, inst["edge"].shape[1], obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (S, 1)))
    f4, _, fi = env.replay(torch.as_tensor(seqs, device=env.device), torch.as_tensor(src, device=env.device))
    assert bool((fi == -1).all())
    out = f4.cpu().numpy()
    env.close()
    return out


def _weakly_dominated(p, front):
    return bool((front <= p).all(axis=1).any())


def _check_archive(inst, start_acts, out, local_optimum):
    S = inst["t"].shape[0]
    cnt = out["count"]
    assert (cnt >= 1).all()
    s_idx = np.concatenate([np.full(c, s) for s, c in enumerate(cnt)])
    a_idx = np.concatenate([np.arange(c) for c in cnt])
    # every member's costs are what a plain replay of its actions gives
    np.testing.assert_array_equal(_replay_plain(inst, out["actions"][:, s_idx, a_idx], s_idx.astype(np.int32)),
                                  out["final4"][s_idx, a_idx])
    assert np.isnan(out["final4"][~(np.arange(out["final4"].shape[1])[None] < cnt[:, None])]).all()
    start_f4 = _replay_plain(inst, start_acts.reshape(start_acts.shape[0], -1, 2),
                             np.tile(np.arange(S, dtype=np.int32), start_acts.shape[1]))
    start_obj = pareto.objectives(start_f4).reshape(-1, S, 3)
    for s in range(S):
        fr = out["objectives"][s, :cnt[s]]
        seg = np.array([0, cnt[s]])
        assert pareto.pareto_filter_reference(fr, seg).all()                 # mutually non-dominated, no duplicates
        for p in start_obj[:, s]:
            assert _weakly_dominated(p, fr)
    h = out["hypervolume"]
    assert h.shape == (out["truncated"].shape[0] + 1, S)
    # the archive's region never shrinks; its FP64 volume may move by rounding when a neighbour replaces a member whose
    # costs differ by an ulp (the same schedule's energy summed in another order)
    drop = np.diff(h, axis=0)
    assert (drop >= -1e-12 * h[1:]).all(), drop.min()
    assert out["replays"] >= start_acts.shape[1] * S
    if local_optimum:
        assert out["explored"][np.arange(out["explored"].shape[1])[None] < cnt[:, None]].all()
        # every neighbour of every member, filtered after the archive: none survives
        members = torch.as_tensor(out["actions"][:, s_idx, a_idx])
        moves = search.neighbour_moves(members, torch.as_tensor(inst["t"][s_idx]))
        nb = search.apply_moves(members, moves).numpy()
        nb_inst = s_idx[moves[:, 0].numpy()]
        nf4 = _replay_plain(inst, nb, nb_inst.astype(np.int32))
        for s in range(S):  # the kernel, pinned to the reference in test_pareto.py, at these sizes
            pts = np.concatenate((out["objectives"][s, :cnt[s]], pareto.objectives(nf4[nb_inst == s])))
            keep = pareto.pareto_filter(torch.as_tensor(pts, device="cuda"), [0, len(pts)]).cpu().numpy()
            assert keep[:cnt[s]].all() and not keep[cnt[s]:].any()


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(3, 4, 2), (4, 3, 2), (2, 5, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_small_sizes_reach_a_pareto_local_optimum(size):
    J, M, E = size
    inst, acts = _start(J, M, E, 4, 3, seed=11)
    out = search.pareto_local_search(inst, acts, rounds=500, expand=4)
    assert out["hypervolume"].shape[0] - 1 < 500 and not out["truncated"].any()
    _check_archive(inst, acts, out, local_optimum=True)


@pytest.mark.gpu
def test_shipped_instances_reach_a_pareto_local_optimum():
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    pick = np.array([0, 17])
    inst = {k: g[k][pick] for k in ("t", "p", "transT", "edge")}
    rand = _start(6, 6, 2, 2, 2, seed=4, d=inst)[1]
    out = search.pareto_local_search(inst, rand, rounds=2000, expand=32, max_archive=4096)
    assert out["hypervolume"].shape[0] - 1 < 2000 and not out["truncated"].any()
    _check_archive(inst, rand, out, local_optimum=True)
    assert (out["hypervolume"][-1] > out["hypervolume"][0]).all()


@pytest.mark.gpu
def test_deterministic_and_independent_of_chunking_and_batch():
    inst, acts = _start(6, 6, 2, 5, 2, seed=31)
    kw = dict(rounds=4, expand=3, max_archive=64)
    a = search.pareto_local_search(inst, acts, **kw)
    b = search.pareto_local_search(inst, acts, **kw)
    c = search.pareto_local_search(inst, torch.as_tensor(acts), max_candidates=173, **kw)
    for k in KEYS:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        np.testing.assert_array_equal(a[k], c[k], err_msg=k)
    assert a["replays"] == b["replays"] == c["replays"]
    pick = np.array([3, 0, 4])
    d = search.pareto_local_search({k: v[pick] for k, v in inst.items()}, acts[:, :, pick], **kw)
    r = d["hypervolume"].shape[0]
    assert r <= a["hypervolume"].shape[0]
    np.testing.assert_array_equal(d["hypervolume"], a["hypervolume"][:r, pick])
    if r == a["hypervolume"].shape[0]:
        for k in ("actions", "final4", "count", "explored"):
            np.testing.assert_array_equal(d[k], np.take(a[k], pick, axis=1 if k == "actions" else 0), err_msg=k)
    # a single start sequence per instance: the [N,S,2] form equals K = 1
    e = search.pareto_local_search(inst, acts[:, 0], **kw)
    f = search.pareto_local_search(inst, acts[:, :1], **kw)
    for k in KEYS:
        np.testing.assert_array_equal(e[k], f[k], err_msg=k)


@pytest.mark.gpu
def test_truncation_caps_the_archive():
    inst, acts = _start(6, 6, 2, 3, 4, seed=8)
    out = search.pareto_local_search(inst, acts, rounds=6, expand=4, max_archive=5)
    assert out["truncated"].any() and (out["count"] <= 5).all()
    for s in range(3):
        fr = out["objectives"][s, :out["count"][s]]
        assert pareto.pareto_filter_reference(fr, [0, len(fr)]).all()
    np.testing.assert_array_equal(out["actions"].shape, (36, 3, 5, 2))


@pytest.mark.gpu
def test_invalid_start_raises():
    inst, acts = _start(3, 4, 2, 2, 1, seed=2)
    bad = acts.copy()
    bad[1, 0, 1] = bad[0, 0, 1]
    with pytest.raises(ValueError):
        search.pareto_local_search(inst, bad)
