"""search.py: the single-move neighbourhood (CPU, against a brute force and the CPU oracle) and the steepest-descent
local search on mtfjsp_replay (GPU: round 1 against stepping every neighbour, monotone history, returned actions
stepped plainly, determinism, independence of chunking and batch, and an improvement over greedy on the shipped
instances)."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
from oracle.mtfjsp_oracle import OracleEnv  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SMALL = [(3, 4, 2), (4, 3, 2), (2, 5, 3)]


def _random_sequences(J, M, E, S, seed, left_shift=True):
    d = ins.synthetic_instances(0, S, J, M, E, seed=seed)
    ora = OracleEnv(S, J, M, E, left_shift=left_shift)
    ora.load(d["t"], d["p"], d["transT"], d["edge"])
    ora.scaler_init()
    ora.reset(ins.random_weights(0, S, seed=seed))
    acts = ora.rollout_random(J * M, seed, record_actions=True)["actions"]
    assert (acts >= 0).all()
    return d, acts


def _brute_moves(acts, t):
    """Every single reassignment and insertion, by definition: a feasible other machine; or entry s removed and put
    at index s' (not s, not s-1) of the rest, kept only if every job's ops stay in order."""
    N, S, _ = acts.shape
    M = t.shape[2]
    out = []
    for i in range(S):
        seq = [tuple(x) for x in acts[:, i]]
        for s, (o, m) in enumerate(seq):
            for m2 in range(M):
                if t[i, o, m2] >= 0 and m2 != m:
                    out.append((i, 0, s, m2, seq[:s] + [(o, m2)] + seq[s + 1:]))
        for s in range(N):
            rest = seq[:s] + seq[s + 1:]
            for s2 in range(N):
                if s2 in (s, s - 1):
                    continue
                new = rest[:s2] + [seq[s]] + rest[s2:]
                ops = [o for o, _ in new]
                if all(ops.index(j * M + k) < ops.index(j * M + k + 1) for j in range(N // M) for k in range(M - 1)):
                    out.append((i, 1, s, s2, new))
    return out


@pytest.mark.parametrize("size", SMALL, ids=lambda s: "J%dM%dE%d" % s)
def test_neighbour_moves_equal_brute_force(size):
    J, M, E = size
    d, acts = _random_sequences(J, M, E, 3, seed=11)
    moves = search.neighbour_moves(torch.as_tensor(acts), torch.as_tensor(d["t"]))
    brute = _brute_moves(acts, d["t"])
    assert moves.dtype == torch.int64 and moves.shape == (len(brute), 4)
    np.testing.assert_array_equal(moves.numpy(), np.array([b[:4] for b in brute]))
    nb = search.apply_moves(torch.as_tensor(acts), moves)
    assert nb.dtype == torch.int32 and nb.shape == (J * M, len(brute), 2)
    np.testing.assert_array_equal(nb.numpy(), np.array([b[4] for b in brute]).transpose(1, 0, 2))


@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SMALL + [(6, 6, 2)], ids=lambda s: "J%dM%dE%d" % s)
def test_every_neighbour_steps_validly_and_none_repeats(size, left_shift):
    J, M, E = size
    N = J * M
    d, acts = _random_sequences(J, M, E, 2, seed=5, left_shift=left_shift)
    moves = search.neighbour_moves(torch.as_tensor(acts), torch.as_tensor(d["t"]))
    nb = search.apply_moves(torch.as_tensor(acts), moves).numpy()
    R = nb.shape[1]
    inst = moves[:, 0].numpy()
    ora = OracleEnv(R, J, M, E, left_shift=left_shift)
    ora.load(*(np.asarray(d[k])[inst] for k in ("t", "p", "transT", "edge")))
    ora.scaler_init()
    ora.reset(np.tile([0.4, 0.4, 0.2], (R, 1)))
    for s in range(N):
        _, _, _, inv = ora.step(nb[s, :, 0], nb[s, :, 1])
        assert not inv.any(), s
    for i in range(2):
        seqs = nb[:, inst == i].transpose(1, 0, 2).reshape(-1, 2 * N)
        assert len({r.tobytes() for r in seqs}) == len(seqs)
        assert not (seqs == acts[:, i].reshape(-1)).all(axis=1).any()  # the incumbent is not its own neighbour


def test_sampled_neighbourhood_size_and_determinism():
    d, acts = _random_sequences(6, 6, 2, 4, seed=3)
    a, t = torch.as_tensor(acts), torch.as_tensor(d["t"])
    full = search.neighbour_moves(a, t)
    count = torch.bincount(full[:, 0], minlength=4)
    K = int(count.min()) // 2
    sub = search.neighbour_moves(a, t, max_neighbours=K, seed=1, round_=2)
    np.testing.assert_array_equal(torch.bincount(sub[:, 0], minlength=4).numpy(), np.minimum(count.numpy(), K))
    # a subset of the full list, in its order, without repeats
    key = lambda m: m[:, 0] * 10**9 + m[:, 1] * 10**8 + m[:, 2] * 10**4 + m[:, 3]
    kf, ks = key(full).numpy(), key(sub).numpy()
    assert np.isin(ks, kf).all() and (np.diff(np.searchsorted(kf, ks)) > 0).all()
    np.testing.assert_array_equal(sub.numpy(), search.neighbour_moves(a, t, max_neighbours=K, seed=1, round_=2).numpy())
    other = search.neighbour_moves(a, t, max_neighbours=K, seed=1, round_=3)
    assert other.shape == sub.shape and not torch.equal(other, sub)
    big = search.neighbour_moves(a, t, max_neighbours=int(count.max()), seed=1)
    np.testing.assert_array_equal(big.numpy(), full.numpy())


# ---------------------------------------------------------------------------------------------------------------- GPU
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")


def _step_all(inst, seqs, left_shift, weights=(0.4, 0.4, 0.2)):
    """final4 of [N,R,2] sequences of `inst` stepped plainly from a fresh reset."""
    N, R, _ = seqs.shape
    M = inst["t"].shape[2]
    env = envm.BatchedMTFJSPEnv(R, N // M, M, inst["edge"].shape[1], left_shift=left_shift, weights=weights)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (R, 1)))
    sq = torch.as_tensor(np.asarray(seqs), device=env.device, dtype=torch.int32)
    for s in range(N):
        env.step(sq[s, :, 0].contiguous(), sq[s, :, 1].contiguous())
    assert not bool(env.invalid.any()) and bool(env.done.all())
    return env.costs().cpu().numpy()


def _objective(f4, w=(0.4, 0.4, 0.2)):
    return w[0] * f4[..., 0] + w[1] * (f4[..., 1] + f4[..., 3]) + w[2] * f4[..., 2]


def _gpu_start(J, M, E, S, seed, left_shift=True):
    d, acts = _random_sequences(J, M, E, S, seed, left_shift=left_shift)
    return {k: np.asarray(v) for k, v in d.items()}, acts


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
def test_round_one_equals_stepping_every_neighbour(left_shift):
    inst, acts = _gpu_start(6, 6, 2, 5, seed=21, left_shift=left_shift)
    out = search.local_search(inst, acts, left_shift=left_shift, rounds=1)
    moves = search.neighbour_moves(torch.as_tensor(acts), torch.as_tensor(inst["t"]))
    nb = search.apply_moves(torch.as_tensor(acts), moves).numpy()
    sub = {k: v[moves[:, 0].numpy()] for k, v in inst.items()}
    f4 = _step_all(sub, nb, left_shift)
    obj = _objective(f4)
    start = _objective(_step_all(inst, acts, left_shift))
    np.testing.assert_array_equal(out["history"][0], start)
    exp_actions, exp_obj = acts.copy(), start.copy()
    for i in range(5):
        sel = np.nonzero(moves[:, 0].numpy() == i)[0]
        j = sel[np.argmin(obj[sel])]  # argmin takes the first of equal values: the lowest move index
        if obj[j] < start[i]:
            exp_actions[:, i] = nb[:, j]
            exp_obj[i] = obj[j]
    np.testing.assert_array_equal(out["accepted"][0], exp_obj < start)
    np.testing.assert_array_equal(out["objective"], exp_obj)
    np.testing.assert_array_equal(out["actions"], exp_actions)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (10, 10, 3), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_descent_is_monotone_deterministic_and_replays_plainly(size):
    J, M, E = size
    inst, acts = _gpu_start(J, M, E, 4, seed=8)
    kw = dict(rounds=3 if J * M > 100 else 6, max_neighbours=None if J * M <= 100 else 400, seed=2)
    a = search.local_search(inst, acts, **kw)
    b = search.local_search(inst, acts, **kw)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    h = a["history"]
    assert h.shape[0] == a["accepted"].shape[0] + 1
    assert (np.diff(h, axis=0) <= 0).all()
    np.testing.assert_array_equal((np.diff(h, axis=0) < 0), a["accepted"])
    np.testing.assert_array_equal(h[-1], a["objective"])
    np.testing.assert_array_equal(_step_all(inst, a["actions"], True), a["final4"])
    np.testing.assert_array_equal(_objective(a["final4"]), a["objective"])


@pytest.mark.gpu
def test_full_neighbourhood_result_does_not_depend_on_chunking_or_batch():
    inst, acts = _gpu_start(6, 6, 2, 6, seed=31)
    a = search.local_search(inst, acts, rounds=4)
    b = search.local_search(inst, acts, rounds=4, max_candidates=97)
    for k in ("actions", "final4", "objective"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    # instances 1, 3, 4 alone (in another order): their rows of the joint run, over the rounds those rows moved in
    pick = np.array([4, 1, 3])
    c = search.local_search({k: v[pick] for k, v in inst.items()}, acts[:, pick], rounds=4)
    np.testing.assert_array_equal(c["history"], a["history"][:, pick][: c["history"].shape[0]])
    if c["history"].shape[0] == a["history"].shape[0]:
        np.testing.assert_array_equal(c["actions"], a["actions"][:, pick])


@pytest.mark.gpu
def test_local_search_improves_greedy_on_the_shipped_instances():
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k] for k in ("t", "p", "transT", "edge")}
    op_sd, mch_sd = val.load_actor_state_dicts(os.path.join(GOLD, "policy_golden.npz"), "iotj")
    ja = enc.JobActor(op_sd, 6, 6, precision="tf32")
    ma = enc.MachineActor(mch_sd, 6, precision="tf32")
    gr = val.greedy_validate(ja, ma, inst, return_actions=True)
    out = search.local_search(inst, gr["actions"], rounds=20)
    np.testing.assert_array_equal(out["history"][0], gr["objective"])
    assert (out["objective"] <= gr["objective"]).all()
    assert out["objective"].mean() < gr["objective"].mean()
