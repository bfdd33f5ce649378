"""search.mcts_search and its two kernels.  On the CPU: the exported entry points and their argument errors, mcts_search's
ValueErrors, and mcts_reference on a hand-built 3-job instance (children expanded in flat-index order, a selection by a
score worked out by hand, virtual visits spreading the paths of a round, a full pool stopping expansion).  On the GPU:
mtfjsp_mcts_select / mtfjsp_mcts_backup against mcts_reference bit for bit over scripted rounds, padded completions
against unpadded ones at each row's own depth, and mcts_search's guarantees on the shipped J6M6 instances."""
import ctypes as C
import importlib
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
validate = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
_lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

PDR = os.path.join(os.path.dirname(__file__), "golden", "pdr_golden.npz")
W = (0.4, 0.4, 0.2)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_entry_points_exported_and_argument_errors():
    lib = _lib.lib()
    assert hasattr(lib, "mtfjsp_mcts_select") and hasattr(lib, "mtfjsp_mcts_backup")
    v = C.c_void_p(16)

    def sel(t=v, S=1, J=6, M=6, L=1, P=8, D=36, node=v):
        return lib.mtfjsp_mcts_select(t, None, S, J, M, v, L, P, D, 1.0, node, v, v, v, v, v, v, v, None)

    for kw in ({"t": None}, {"node": None}, {"S": 0}, {"L": 0}, {"P": 0}, {"D": -1}, {"J": 0}, {"M": 1}, {"M": 65},
               {"J": 600, "M": 20}):
        assert sel(**kw) == -1, kw
        assert b"mtfjsp_mcts_select" in lib.mtfjsp_last_error()
    assert lib.mtfjsp_mcts_backup(1, 1, 8, None, v, v, v, v, v, v, None) == -1
    assert lib.mtfjsp_mcts_backup(0, 1, 8, v, v, v, v, v, v, v, None) == -1
    assert lib.mtfjsp_mcts_backup(1, 0, 8, v, v, v, v, v, v, v, None) == -1
    assert lib.mtfjsp_mcts_backup(1, 1, 0, v, v, v, v, v, v, v, None) == -1
    assert b"mtfjsp_mcts_backup" in lib.mtfjsp_last_error()


def test_search_argument_errors():
    g = np.load(PDR)
    inst = {k: g[k][:2] for k in ("t", "p", "transT", "edge")}
    for kw in ({"mask_mode": envm.MASK_ESA}, {"base": "random", "candidates": "rule"}, {"simulations": 0},
               {"leaves": 0}, {"max_nodes": 0}, {"candidates": "some"}, {"c": -1.0}):
        with pytest.raises(ValueError):
            search.mcts_search(inst, **kw)


# J = 3, M = 2: op 0 only on machine 0, op 2 on both, op 4 only on machine 1, op 5 only on machine 0; the root's children
# are flat indices 0, 2, 3, 5 = (0, 0), (2, 0), (2, 1), (4, 1)
T3 = np.array([[[3, -1], [2, -1], [2, 4], [1, 1], [-1, 5], [3, -1]]], dtype=np.float64)
ROOT3 = [(0, 0), (2, 0), (2, 1), (4, 1)]


def _hand_tree(max_nodes):
    """Five rounds of one selection: the root, then its four children, scored 10, 12, 8, 9, 11."""
    tree = search.mcts_trees(1, max_nodes, device="numpy")
    return search.mcts_reference(T3, np.zeros((1, 3), np.int32), tree, 1, 1.0, [[10.0], [12.0], [8.0], [9.0], [11.0]])


def test_reference_expands_in_flat_index_order_then_scores():
    paths, depth, leaf, tree = _hand_tree(64)
    assert depth[:, 0].tolist() == [0, 1, 1, 1, 1] and leaf[:, 0].tolist() == [0, 1, 2, 3, 4]
    assert [tuple(paths[r, 0, 0]) for r in range(1, 5)] == ROOT3
    assert (paths[0] == -1).all() and (paths[1:, 0, 1:] == -1).all()
    nd = tree["node"][0]
    assert [tuple(x) for x in nd[1:5, search.OP:search.MACH + 1]] == ROOT3
    assert (nd[1:5, search.PARENT] == 0).all() and (nd[0, search.FIRST], nd[0, search.NCHILD]) == (1, 4)
    assert nd[0, search.VISITS] == 5 and (nd[:, search.VIRTUAL] == 0).all()
    assert tree["vmin"][0, :5].tolist() == [8.0, 12.0, 8.0, 9.0, 11.0]
    assert tree["lohi"][0].tolist() == [8.0, 12.0] and tree["count"][0] == 5
    # a round of two: the root has 5 visits and this path's virtual one; every child n = 1, v = 0, q = (12 - vmin) / 4
    q = [(12.0 - x) / 4.0 for x in (12.0, 8.0, 9.0, 11.0)]
    first = [qi * 1 / 1 + 1.0 * math.sqrt(6) / 2 for qi in q]
    assert int(np.argmax(first)) == 1                                   # child (2, 0): 1 + sqrt(6)/2
    # the second path sees child 2's virtual visit (n = 1, v = 1) and the root's two virtual visits
    second = [q[i] * 1 / (1 + (i == 1)) + math.sqrt(7) / (2 + (i == 1)) for i in range(4)]
    assert int(np.argmax(second)) == 2                                  # child (2, 1): 0.75 + sqrt(7)/2
    p2, d2, l2, t2 = search.mcts_reference(T3, np.zeros((1, 3), np.int32), tree, 2, 1.0, [[7.0, 9.5]])
    # child 2 is expanded on the way (reached before): (2, 0) leaves job 1 at op 3 -> children (0,0), (3,0), (3,1), (4,1)
    assert d2[0].tolist() == [2, 2]
    assert [tuple(x) for x in p2[0, 0, :2]] == [(2, 0), (0, 0)] and [tuple(x) for x in p2[0, 1, :2]] == [(2, 1), (0, 0)]
    nd2 = t2["node"][0]
    assert [tuple(x) for x in nd2[5:9, search.OP:search.MACH + 1]] == [(0, 0), (3, 0), (3, 1), (4, 1)]
    assert l2[0].tolist() == [5, 9] and t2["count"][0] == 13
    assert t2["vmin"][0, [0, 2, 3, 5, 9]].tolist() == [7.0, 7.0, 9.0, 7.0, 9.5]
    assert t2["lohi"][0].tolist() == [7.0, 12.0] and nd2[0, search.VISITS] == 7


def test_reference_full_pool_stops_expansion():
    _, _, _, tree = _hand_tree(5)                                       # the root and its four children fill the pool
    p, d, l, t2 = search.mcts_reference(T3, np.zeros((1, 3), np.int32), tree, 1, 1.0, [[7.0]])
    assert d[0, 0] == 1 and l[0, 0] == 2 and tuple(p[0, 0, 0]) == (2, 0)
    assert t2["count"][0] == 5 and (t2["node"][0, 2, search.FIRST], t2["node"][0, 2, search.NCHILD]) == (-1, 0)
    assert t2["node"][0, 2, search.VISITS] == 2 and t2["vmin"][0, 2] == 7.0


def test_reference_terminal_node_is_scored_again():
    # jobs 0 and 1 finished, job 2 at its last op: the root has one child, (5, 0), which is terminal
    nx = np.array([[2, 2, 1]], np.int32)
    tree = search.mcts_trees(1, 16, device="numpy")
    _, d, l, t2 = search.mcts_reference(T3, nx, tree, 1, 1.0, [[5.0], [4.0], [4.0], [3.0]])
    assert d[:, 0].tolist() == [0, 1, 1, 1] and l[:, 0].tolist() == [0, 1, 1, 1] and t2["count"][0] == 2
    assert t2["node"][0, 1, search.VISITS] == 3 and t2["vmin"][0, 1] == 3.0


# ---------------------------------------------------------------------------------------------------------------- GPU
def _kernel_case(J, M, S, seed):
    rng = np.random.default_rng(seed)
    N = J * M
    t = ins.synthetic_instances(0, S, J, M, 2 if M < 10 else 3, seed=seed)["t"]
    nx = rng.integers(0, M + 1, size=(S, J)).astype(np.int32)
    nx[:, 0] = 0
    nx[0] = 0
    nx[-1, : J // 2] = M                                                  # finished jobs
    mach = np.empty((S, N), np.int32)
    for s in range(S):
        for o in range(N):
            mach[s, o] = rng.choice(np.nonzero(t[s, o] >= 0)[0])
    return t, nx, mach


@pytest.mark.gpu
@pytest.mark.parametrize("J,M,cand,S,P,L,rounds", [(6, 6, "all", 6, 400, 8, 7), (6, 6, "rule", 6, 60, 8, 7),
                                                  (10, 10, "all", 5, 1500, 16, 9), (10, 10, "rule", 5, 200, 8, 7),
                                                  (30, 20, "all", 3, 4000, 64, 12)])
def test_kernels_equal_the_reference(J, M, cand, S, P, L, rounds):
    """Enough selections that every size scores children past the fresh ones (C = 600 at J30M20: 19 lane chunks),
    reaches depth 2 and fills its pool."""
    t, nx, mach = _kernel_case(J, M, S, 11 + J)
    rng = np.random.default_rng(J * M)
    obj = rng.integers(0, 12, size=(rounds, S * L)).astype(np.float64) * 0.25 + 100.0     # many ties
    obj[rng.random(obj.shape) < 0.05] = np.inf
    rule = mach if cand == "rule" else None
    ref_tree = search.mcts_trees(S, P, device="numpy")
    rp, rd, rl, rt = search.mcts_reference(t, nx, ref_tree, L, 0.7, obj, mach=rule)
    tree = search.mcts_trees(S, P)
    dev = tree["node"].device
    td, nxd = torch.as_tensor(t, device=dev), torch.as_tensor(nx, device=dev)
    md = None if rule is None else torch.as_tensor(rule, device=dev)
    for r in range(rounds):
        paths, depth, leaf = search.mcts_select(td, nxd, tree, L, 0.7, md)
        np.testing.assert_array_equal(paths.cpu().numpy(), rp[r], err_msg="paths %d" % r)
        np.testing.assert_array_equal(depth.cpu().numpy(), rd[r], err_msg="depth %d" % r)
        np.testing.assert_array_equal(leaf.cpu().numpy(), rl[r], err_msg="leaf %d" % r)
        search.mcts_backup(tree, leaf, torch.as_tensor(obj[r], device=dev))
    for k in rt:
        np.testing.assert_array_equal(tree[k].cpu().numpy(), rt[k], err_msg=k)
    assert rd.max() >= 2 and (rt["count"] > P - J * M).any()


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [False, True])
@pytest.mark.parametrize("J,M,E", [(6, 6, 2), (13, 11, 3), (30, 20, 5)])
def test_padded_completions_equal_unpadded_ones(J, M, E, left_shift):
    N = J * M
    B = 6
    d = ins.synthetic_instances(0, B, J, M, E, seed=40 + J)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, obs_dtype=torch.float32,
                                mask_mode=envm.MASK_FINISHED)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed=3))
    for _ in range(N // 3):
        env.random_step(seed=9, mask_mode=envm.MASK_FINISHED)
    R = 4 * B
    src = (torch.arange(R, device=env.device) % B).to(torch.int32)
    key, mach = rules.priority_table("MWKR_T", "SPT", d["t"], d["p"], J, M)
    kd, md = torch.as_tensor(key, device=env.device), torch.as_tensor(mach, device=env.device)
    _, _, _, seqs = env.complete(src, base="random", seed=5, mask_mode=envm.MASK_FINISHED)   # valid from the state
    rest = N - N // 3
    depth = torch.as_tensor(np.random.default_rng(J).integers(0, min(rest, 9) + 1, R), device=env.device)
    depth[0] = 0
    T = int(depth.max())
    steps = torch.arange(T, device=env.device)[:, None, None]
    padded = torch.where(steps < depth[None, :, None], seqs[:T], -1)
    for base, kw in (("random", {}), ("priority", {"key": kd, "mach": md})):
        got = env.complete(src, padded, base=base, seed=7, mask_mode=envm.MASK_FINISHED, **kw)
        fi = got[2].cpu().numpy()
        dn = depth.cpu().numpy()
        np.testing.assert_array_equal(fi, np.where(dn < T, dn, -1))
        for dd in np.unique(dn):
            own = env.complete(src, seqs[:dd] if dd else None, base=base, seed=7, mask_mode=envm.MASK_FINISHED, **kw)
            rows = dn == dd
            assert (own[2].cpu().numpy()[rows] == -1).all()
            for a, b, name in ((got[0], own[0], "final4"), (got[1], own[1], "return5"),
                               (got[3].transpose(0, 1), own[3].transpose(0, 1), "base_actions")):
                np.testing.assert_array_equal(a.cpu().numpy()[rows], b.cpu().numpy()[rows], err_msg="%s %s d=%d" %
                                              (base, name, dd))
    env.close()


def _instances(sl):
    g = np.load(PDR)
    return {k: g[k][sl] for k in ("t", "p", "transT", "edge")}, g


def _replay(inst, actions):
    S = inst["t"].shape[0]
    env = envm.BatchedMTFJSPEnv(S, 6, 6, 2, left_shift=False, obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile(list(W), (S, 1)))
    f4, _, fi = env.replay(torch.as_tensor(actions, device=env.device))
    out = f4.cpu().numpy(), fi.cpu().numpy()
    env.close()
    return out


def _check_returned(inst, out):
    f4, fi = _replay(inst, out["actions"])
    assert (fi == -1).all()
    np.testing.assert_array_equal(f4, out["final4"])
    np.testing.assert_array_equal(validate._objective(f4, W), out["objective"])
    assert (out["objective"] <= out["base_objective"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("candidates,sims", [("all", 37), ("rule", 7)])
def test_priority_mcts_guarantees(candidates, sims):
    inst, g = _instances(slice(0, 10))
    rule_obj = validate._objective(g["gold"][[str(x) for x in g["rule_names"]].index("MWKR_T+SPT")][:10], W)
    out = search.mcts_search(inst, base=("MWKR_T", "SPT"), candidates=candidates, simulations=sims, leaves=8)
    h = out["history"]
    assert h.shape == (37, 10) and out["actions"].shape == (36, 10, 2)
    np.testing.assert_array_equal(h[0], rule_obj)
    np.testing.assert_array_equal(out["base_objective"], rule_obj)
    assert (np.diff(h, axis=0) <= 0).all()
    np.testing.assert_array_equal(out["objective"], h.min(0))
    _check_returned(inst, out)
    again = search.mcts_search(inst, base=("MWKR_T", "SPT"), candidates=candidates, simulations=sims, leaves=8)
    one, _ = _instances(slice(4, 5))
    alone = search.mcts_search(one, base=("MWKR_T", "SPT"), candidates=candidates, simulations=sims, leaves=8,
                               max_candidates=3)
    for k in ("actions", "final4", "objective", "history", "nodes"):
        np.testing.assert_array_equal(again[k], out[k], err_msg=k)
        sl = out[k][:, 4:5] if k in ("actions", "history") else out[k][4:5]
        np.testing.assert_array_equal(alone[k], sl, err_msg=k)


@pytest.mark.gpu
def test_small_budget_small_pool_and_random_base():
    inst, _ = _instances(slice(0, 6))
    # one selection a decision never expands a root: every decision follows the base and restarts the tree
    low = search.mcts_search(inst, simulations=1, leaves=1)
    np.testing.assert_array_equal(low["objective"], low["base_objective"])
    assert (np.diff(low["history"], axis=0) == 0).all() and (low["nodes"] == 1).all()
    _check_returned(inst, low)
    tight = search.mcts_search(inst, simulations=24, leaves=8, max_nodes=60)
    assert (tight["nodes"] <= 60).all()
    _check_returned(inst, tight)
    a = search.mcts_search(inst, base="random", simulations=16, leaves=8, seed=3)
    b = search.mcts_search(inst, base="random", simulations=16, leaves=8, seed=3)
    for k in ("actions", "final4", "objective", "history"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    _check_returned(inst, a)
    assert a["completions"] == 6 + 36 * 2 * 6 * 8
