"""search.tabu_search, mtfjsp_tabu_move and search.tabu_reference.  On the CPU: the reference against a brute-force
statement of the rules on forged states (tabu moves, aspiration, ties, NaN objectives, an all-tabu instance, an empty
and a malformed segment, moves of another instance), and the argument errors of the entry point.  On the GPU: the kernel
against the reference over real neighbourhoods and on the forged states, tabu_search against local_search while that
descends, its invariants, and its result on the shipped J6M6 instances."""
import ctypes as C
import importlib
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
validate = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
from oracle.mtfjsp_oracle import OracleEnv  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
W = (0.4, 0.4, 0.2)
E_ARG = -1


def _random_sequences(J, M, E, S, seed, left_shift=True):
    d = ins.synthetic_instances(0, S, J, M, E, seed=seed)
    ora = OracleEnv(S, J, M, E, left_shift=left_shift)
    ora.load(d["t"], d["p"], d["transT"], d["edge"])
    ora.scaler_init()
    ora.reset(ins.random_weights(0, S, seed=seed))
    acts = ora.rollout_random(J * M, seed, record_actions=True)["actions"]
    return {k: np.asarray(v) for k, v in d.items()}, acts


def _brute(state, moves, seg, obj, f4, it, tm, ti):
    """The rules of include/mtfjsp.h stated directly: the admissible (objective, index) pairs, their least, and the move
    applied by search.apply_moves."""
    st = {k: np.array(v, copy=True) for k, v in state.items()}
    S, N, M = st["cur"].shape[0], st["cur"].shape[1], st["mach_until"].shape[2]
    R = len(moves)
    chosen = []
    for s in range(S):
        lo, hi = int(seg[s]), int(seg[s + 1])
        if not 0 <= lo <= hi <= R:
            chosen.append(-2)
            continue
        cand = []
        for r in range(lo, hi):
            i, kind, ms, arg = (int(x) for x in moves[r])
            if i != s or kind not in (0, 1) or not 0 <= ms < N:
                continue
            o, m_old = (int(x) for x in st["cur"][s, ms])
            ok = 0 <= o < N and (0 <= arg < M and 0 <= m_old < M if kind == 0 else 0 <= arg < N)
            if not ok or math.isnan(obj[r]):
                continue
            tabu = st["mach_until"][s, o, arg] > it if kind == 0 else st["op_until"][s, o] > it
            if not tabu or obj[r] < st["best_obj"][s]:
                cand.append((float(obj[r]), r))
        if not cand:
            chosen.append(-1)
            continue
        v, r = min(cand)
        _, kind, ms, arg = (int(x) for x in moves[r])
        o, m_old = (int(x) for x in st["cur"][s, ms])
        one = torch.tensor([[0, kind, ms, arg]])
        st["cur"][s] = search.apply_moves(torch.as_tensor(st["cur"][s][:, None]), one)[:, 0].numpy()
        if kind == 0:
            st["mach_until"][s, o, m_old] = it + 1 + tm
        else:
            st["op_until"][s, o] = it + 1 + ti
        st["cur_obj"][s], st["cur_f4"][s] = obj[r], f4[r]
        if obj[r] < state["best_obj"][s]:
            st["best"][s], st["best_obj"][s], st["best_f4"][s] = st["cur"][s], obj[r], f4[r]
        chosen.append(r)
    return st, np.array(chosen, dtype=np.int32)


def _forged(seed):
    """A tabu state of 8 J2M3 instances with random tables around iteration 5, a move list with ties, NaNs and
    aspiration, and: instance 5 all tabu, instance 6 an empty segment, instance 7 a decreasing segment; a few moves
    carry another instance's field."""
    rng = np.random.default_rng(seed)
    J, M, S, it = 2, 3, 8, 5
    N = J * M
    d, acts = _random_sequences(J, M, 1, S, seed=seed + 1)
    moves = search.neighbour_moves(torch.as_tensor(acts), torch.as_tensor(d["t"])).numpy()
    moves = moves[moves[:, 0] != 6]
    f4 = rng.integers(0, 4, size=(S, 4)).astype(np.float64)
    st = search.tabu_state(np.ascontiguousarray(acts.transpose(1, 0, 2)).astype(np.int32), f4, W, M)
    st["best_obj"] = st["cur_obj"] - rng.integers(0, 3, size=S)               # best at or below cur
    st["mach_until"] = rng.integers(it - 2, it + 3, size=(S, N, M)).astype(np.int32)
    st["op_until"] = rng.integers(it - 2, it + 3, size=(S, N)).astype(np.int32)
    st["mach_until"][5], st["op_until"][5] = it + 1, it + 1
    R = moves.shape[0]
    obj = rng.integers(0, 6, size=R).astype(np.float64)                       # small integers: many ties
    obj[rng.random(R) < 0.1] = np.nan
    obj[moves[:, 0] == 5] = st["best_obj"][5] + rng.integers(0, 3, size=int((moves[:, 0] == 5).sum()))
    mf4 = rng.random((R, 4))
    wrong = np.nonzero(rng.random(R) < 0.05)[0]
    moves[wrong, 0] = (moves[wrong, 0] + 1) % S
    inst = moves[:, 0].copy()
    inst[wrong] = (inst[wrong] - 1) % S                                        # the segment a move sits in
    seg = np.concatenate(([0], np.cumsum(np.bincount(inst, minlength=S)))).astype(np.int64)
    seg[8] = seg[7] - 1                                                        # instance 7: seg[8] < seg[7]
    return st, moves.astype(np.int32), seg, obj, mf4, it


def test_reference_equals_the_rules_on_forged_states():
    for seed in range(6):
        st, moves, seg, obj, mf4, it = _forged(seed)
        for tm, ti in ((3, 2), (0, 0)):
            got, ch = search.tabu_reference(st, moves, seg, obj, mf4, it, tm, ti)
            exp, ch2 = _brute(st, moves, seg, obj, mf4, it, tm, ti)
            np.testing.assert_array_equal(ch, ch2)
            for k in st:
                np.testing.assert_array_equal(got[k], exp[k], err_msg="seed %d %s" % (seed, k))
            assert ch[5] == -1 and ch[6] == -1 and ch[7] == -2
            for k in st:
                np.testing.assert_array_equal(got[k][5:], st[k][5:])           # instances that stay put
        # some instance moves below its best
        taken = ch[ch >= 0]
        assert (obj[taken] < st["best_obj"][np.nonzero(ch >= 0)[0]]).any()


def test_reference_ties_go_to_the_lowest_index_and_nan_never_wins():
    st, moves, seg, obj, mf4, it = _forged(11)
    st["mach_until"][:], st["op_until"][:] = 0, 0                              # nothing tabu
    lo, hi = int(seg[0]), int(seg[1])
    moves[lo:hi, 0] = 0
    obj[:] = 9.0
    obj[lo] = np.nan
    obj[lo + 2] = obj[lo + 4] = 1.0
    _, ch = search.tabu_reference(st, moves, seg, obj, mf4, it)
    assert ch[0] == lo + 2
    obj[lo:hi] = np.nan
    _, ch = search.tabu_reference(st, moves, seg, obj, mf4, it)
    assert ch[0] == -1


def test_tabu_move_argument_errors_name_the_entry_point():
    lib = libm.lib()
    v = C.c_void_p(16)  # never dereferenced: every argument error is found before any launch

    def call(S=2, J=2, M=3, moves=v, R=4, seg=v, obj=v, f4=v, it=0, tm=1, ti=1, state=(v,) * 8, chosen=v):
        return lib.mtfjsp_tabu_move(S, J, M, moves, R, seg, obj, f4, it, tm, ti, *state, chosen, None)

    bad = [{"S": 0}, {"J": 0}, {"M": 1}, {"M": 65}, {"J": 600, "M": 20}, {"R": -1}, {"R": 1 << 31}, {"moves": None},
           {"obj": None}, {"f4": None}, {"seg": None}, {"chosen": None}, {"it": -1}, {"tm": -1}, {"ti": -1},
           {"it": 2**31 - 2, "tm": 1}, {"it": 2**31 - 2, "ti": 5}]
    bad += [{"state": tuple(None if j == i else v for j in range(8))} for i in range(8)]
    for kw in bad:
        assert call(**kw) == E_ARG, kw
        assert b"mtfjsp_tabu_move" in lib.mtfjsp_last_error()


def test_search_argument_errors():
    d, acts = _random_sequences(3, 4, 2, 2, seed=1)
    for kw in ({"max_candidates": 0}, {"iterations": -1}, {"tenure_mach": -1}, {"tenure_ins": -2}):
        with pytest.raises(ValueError):
            search.tabu_search(d, acts, **kw)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _to_dev(st, dev):
    return {k: torch.as_tensor(v, device=dev) for k, v in st.items()}


def _assert_state(dev_st, ref_st, where):
    for k in ref_st:
        np.testing.assert_array_equal(dev_st[k].cpu().numpy(), ref_st[k], err_msg="%s %s" % (where, k))


@pytest.mark.gpu
def test_kernel_equals_reference_on_forged_states():
    dev = torch.device("cuda", torch.cuda.current_device())
    for seed in range(4):
        st, moves, seg, obj, mf4, it = _forged(seed)
        for tm, ti in ((3, 2), (0, 0)):
            ref, rch = search.tabu_reference(st, moves, seg, obj, mf4, it, tm, ti)
            ds = _to_dev(st, dev)
            ch = search.tabu_move(ds, torch.as_tensor(moves, device=dev), torch.as_tensor(seg, device=dev),
                                  torch.as_tensor(obj, device=dev), torch.as_tensor(mf4, device=dev), it, tm, ti)
            np.testing.assert_array_equal(ch.cpu().numpy(), rch)
            _assert_state(ds, ref, "seed %d" % seed)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (10, 10, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_kernel_equals_reference_over_real_neighbourhoods(size):
    J, M, E = size
    S, N = 4, J * M
    d, acts = _random_sequences(J, M, E, S, seed=J)
    env = envm.BatchedMTFJSPEnv(S, J, M, E, weights=W, obs_dtype=torch.float32)
    dev = env.device
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(W), (S, 1)))
    cur = torch.as_tensor(acts, device=dev, dtype=torch.int32)
    f4, _, _ = env.replay(cur)
    ds = search.tabu_state(cur.transpose(0, 1).contiguous(), f4, W, M)
    ref = {k: v.cpu().numpy() for k, v in ds.items()}
    t = torch.as_tensor(d["t"], device=dev)
    taken = 0
    for it in range(20):
        base = ds["cur"].transpose(0, 1)
        moves = search.neighbour_moves(base, t, None if N <= 36 else 300, 5, it)
        mf4, _, fi = env.replay_moves(base, moves)
        assert (fi == -1).all()
        obj = validate._objective(mf4, W)
        seg = torch.cat((torch.zeros(1, dtype=torch.int64, device=dev),
                         torch.cumsum(torch.bincount(moves[:, 0], minlength=S), 0)))
        ch = search.tabu_move(ds, moves, seg, obj, mf4, it, 2, 3)
        ref, rch = search.tabu_reference(ref, moves.cpu().numpy(), seg.cpu().numpy(), obj.cpu().numpy(),
                                         mf4.cpu().numpy(), it, 2, 3)
        np.testing.assert_array_equal(ch.cpu().numpy(), rch, err_msg="iteration %d" % it)
        _assert_state(ds, ref, "iteration %d" % it)
        taken += int((rch >= 0).sum())
    assert taken == 20 * S


def _step_all(inst, seqs, left_shift):
    N, R, _ = seqs.shape
    M = inst["t"].shape[2]
    env = envm.BatchedMTFJSPEnv(R, N // M, M, inst["edge"].shape[1], left_shift=left_shift, weights=W)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile(np.asarray(W), (R, 1)))
    sq = torch.as_tensor(np.asarray(seqs), device=env.device, dtype=torch.int32)
    for s in range(N):
        env.step(sq[s, :, 0].contiguous(), sq[s, :, 1].contiguous())
    assert not bool(env.invalid.any()) and bool(env.done.all())
    return env.costs().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
def test_tabu_follows_local_search_while_it_descends(left_shift):
    inst, acts = _random_sequences(6, 6, 2, 6, seed=41, left_shift=left_shift)
    ls = search.local_search(inst, acts, left_shift=left_shift, rounds=200)
    a = ls["accepted"].sum(0)
    assert ls["accepted"].shape[0] < 200                                       # local_search reached its optimum
    tb = search.tabu_search(inst, acts, left_shift=left_shift, iterations=int(a.max()) + 5)
    for i in range(6):
        np.testing.assert_array_equal(tb["history"][: a[i] + 1, i], ls["history"][: a[i] + 1, i], err_msg=str(i))
    assert (tb["objective"] <= ls["objective"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (10, 10, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_invariants_and_determinism(size):
    J, M, E = size
    inst, acts = _random_sequences(J, M, E, 4, seed=8)
    kw = dict(iterations=15, max_neighbours=None if J * M <= 36 else 300, seed=2, tenure_mach=3, tenure_ins=4)
    a = search.tabu_search(inst, acts, **kw)
    b = search.tabu_search(inst, acts, **kw)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    h, bh = a["history"], a["best_history"]
    assert h.shape == bh.shape == (16, 4) and a["chosen"].shape == (15, 4)
    assert (np.diff(bh, axis=0) <= 0).all()
    np.testing.assert_array_equal(bh, np.minimum.accumulate(h, axis=0))
    np.testing.assert_array_equal(bh[-1], a["objective"])
    np.testing.assert_array_equal(_step_all(inst, a["actions"], True), a["final4"])
    np.testing.assert_array_equal(validate._objective(a["final4"], W), a["objective"])


@pytest.mark.gpu
def test_result_does_not_depend_on_chunking_or_batch():
    inst, acts = _random_sequences(6, 6, 2, 6, seed=31)
    a = search.tabu_search(inst, acts, iterations=30)
    b = search.tabu_search(inst, acts, iterations=30, max_candidates=97)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    pick = np.array([4, 1, 3])
    c = search.tabu_search({k: v[pick] for k, v in inst.items()}, acts[:, pick], iterations=30)
    for k in ("history", "best_history", "objective", "final4"):
        np.testing.assert_array_equal(c[k], a[k][..., pick, :] if k == "final4" else a[k][..., pick], err_msg=k)
    np.testing.assert_array_equal(c["actions"], a["actions"][:, pick])


@pytest.mark.gpu
def test_tabu_beats_local_search_from_greedy_on_the_shipped_instances():
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: g[k] for k in ("t", "p", "transT", "edge")}
    op_sd, mch_sd = validate.load_actor_state_dicts(os.path.join(GOLD, "policy_golden.npz"), "iotj")
    ja = enc.JobActor(op_sd, 6, 6, precision="tf32")
    ma = enc.MachineActor(mch_sd, 6, precision="tf32")
    gr = validate.greedy_validate(ja, ma, inst, return_actions=True)
    ls = search.local_search(inst, gr["actions"], rounds=200)
    assert ls["accepted"].shape[0] < 60
    tb = search.tabu_search(inst, gr["actions"], iterations=60)
    np.testing.assert_array_equal(tb["history"][0], gr["objective"])
    assert (tb["objective"] <= ls["objective"]).all()
    assert tb["objective"].mean() < ls["objective"].mean()
