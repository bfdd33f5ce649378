"""mtfjsp_replay_moves / BatchedMTFJSPEnv.replay_moves: single-move neighbours replayed from their base sequence and the
move list, without building them.  On the CPU: the argument errors.  On the GPU: bit equality with
replay(apply_moves(...)) on whole neighbourhoods at specialised, unspecialised and edge sizes, with and without left
shift, on sampled J30M20 neighbourhoods, with permuted and duplicated base sources (Q != B), and on moves that are
well-formed but replay an invalid action; every kind of malformed move; and a handle the call leaves untouched."""
import ctypes as C
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

E_ARG, E_STATE = -1, -3
B = 3
SIZES = [(3, 4, 2), (6, 6, 2), (10, 10, 3), (13, 11, 3), (1, 2, 1), (2, 64, 64), (70, 2, 1)]


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_argument_errors_name_the_entry_point():
    lib = libm.lib()
    v = C.c_void_p(16)  # never dereferenced: every argument error is found before the handle is read

    def call(h=v, src=v, Q=2, base=v, moves=v, R=5):
        return lib.mtfjsp_replay_moves(h, src, Q, base, moves, R, v, v, v, None)

    for kw in ({"h": None}, {"src": None}, {"base": None}, {"moves": None}, {"Q": 0}, {"Q": -1}, {"R": 0}, {"R": -3}):
        assert call(**kw) == E_ARG, kw
        assert b"mtfjsp_replay_moves" in lib.mtfjsp_last_error()


# ---------------------------------------------------------------------------------------------------------------- GPU
def _env(J, M, E, d, left_shift, B_=B):
    env = envm.BatchedMTFJSPEnv(B_, J, M, E, left_shift=left_shift, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (B_, 1)))
    return env


def _random_sequences(J, M, E, seed, left_shift):
    """Instances and one complete random valid sequence per env ([N,B,2] int32 on the device), from a second handle."""
    d = ins.synthetic_instances(0, B, J, M, E, seed=seed)
    gen = _env(J, M, E, d, left_shift)
    gen.obs()
    acts = []
    for _ in range(J * M):
        gen.random_step(seed=seed)
        acts.append(torch.stack((gen.op, gen.mach), 1).clone())
    gen.close()
    return d, torch.stack(acts)


def _assert_same(got, exp, where):
    for name, g, e in zip(("final4", "return5", "first_invalid"), got, exp):
        np.testing.assert_array_equal(g.cpu().numpy(), e.cpu().numpy(), err_msg="%s %s" % (where, name))


def _materialised(env, base, moves, base_src):
    return env.replay(search.apply_moves(base, moves), base_src[moves[:, 0]].to(torch.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_whole_neighbourhood_equals_replay_of_the_built_neighbours(size, left_shift):
    J, M, E = size
    d, acts = _random_sequences(J, M, E, 50 + J, left_shift)
    env = _env(J, M, E, d, left_shift)
    t = torch.as_tensor(d["t"], device=env.device)
    moves = search.neighbour_moves(acts, t)
    assert moves.shape[0] > 0
    src = torch.arange(B, device=env.device)
    got = env.replay_moves(acts, moves)
    _assert_same(got, _materialised(env, acts, moves, src), "full")
    assert (got[2] == -1).all()


@pytest.mark.gpu
def test_sampled_neighbourhood_at_j30m20():
    J, M, E = 30, 20, 5
    d, acts = _random_sequences(J, M, E, 77, True)
    env = _env(J, M, E, d, True)
    moves = search.neighbour_moves(acts, torch.as_tensor(d["t"], device=env.device), max_neighbours=300, seed=4)
    assert moves.shape[0] == 3 * 300
    _assert_same(env.replay_moves(acts, moves), _materialised(env, acts, moves, torch.arange(B, device=env.device)),
                 "sampled")


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_permuted_and_duplicated_base_sources(size):
    J, M, E = size
    d, acts = _random_sequences(J, M, E, 9, True)
    env = _env(J, M, E, d, True)
    idx = torch.tensor([2, 0, 0, 1, 2, 2, 1], device=env.device)               # Q = 7 rows of B = 3 envs
    base = acts.index_select(1, idx)
    t = torch.as_tensor(d["t"], device=env.device)
    moves = search.neighbour_moves(base, t[idx], max_neighbours=150, seed=1)
    _assert_same(env.replay_moves(base, moves, idx), _materialised(env, base, moves, idx), "Q=7")
    one = env.replay_moves(base[:, 3:4], moves[moves[:, 0] == 3] - torch.tensor([3, 0, 0, 0], device=env.device),
                           idx[3:4])                                           # Q = 1 < B
    _assert_same(one, [x[moves[:, 0] == 3] for x in env.replay_moves(base, moves, idx)], "Q=1")


@pytest.mark.gpu
def test_well_formed_moves_that_replay_an_invalid_action():
    J, M, E = 6, 6, 2
    N = J * M
    d, acts = _random_sequences(J, M, E, 13, True)
    env = _env(J, M, E, d, True)
    dev = env.device
    t = d["t"]
    mv = []
    for i in range(B):
        for s in range(0, N, 5):
            o = int(acts[s, i, 0])
            bad_m = [m for m in range(M) if t[i, o, m] < 0]
            mv += [(i, 0, s, bad_m[0] if bad_m else M), (i, 0, s, -1), (i, 0, s, M + 3)]   # infeasible / out of range
            mv += [(i, 1, s, 0), (i, 1, s, N - 1)]                             # usually breaks job order
    moves = torch.tensor(mv, device=dev)
    src = torch.arange(B, device=dev)
    got = env.replay_moves(acts, moves)
    _assert_same(got, _materialised(env, acts, moves, src), "invalid")
    assert (got[2][moves[:, 1] == 0] >= 0).all()


@pytest.mark.gpu
def test_malformed_moves_are_rows_of_zeros():
    J, M, E = 6, 6, 2
    N = J * M
    d, acts = _random_sequences(J, M, E, 21, True)
    env = _env(J, M, E, d, True)
    dev = env.device
    base = torch.cat((acts, acts[:, :1]), 1)                                   # Q = 4; row 3's source is out of range
    src = torch.tensor([0, 1, 2, B], dtype=torch.int32, device=dev)
    good = search.neighbour_moves(acts, torch.as_tensor(d["t"], device=dev), max_neighbours=20, seed=3)
    bad = torch.tensor([(-1, 0, 1, 1), (4, 1, 2, 5), (0, 2, 1, 1), (1, -1, 1, 1), (2, 0, -1, 1), (0, 0, N, 1),
                        (1, 1, 3, -1), (2, 1, 3, N), (0, 1, -2, 4), (3, 0, 1, 1), (3, 1, 4, 9)], device=dev)
    at = torch.arange(bad.shape[0], device=dev) * 3 + 1                         # each between two good moves
    mixed = torch.empty((good.shape[0] + bad.shape[0], 4), dtype=good.dtype, device=dev)
    is_bad = torch.zeros(mixed.shape[0], dtype=torch.bool, device=dev)
    is_bad[at] = True
    mixed[is_bad] = bad
    mixed[~is_bad] = good
    got = env.replay_moves(base, mixed, src)
    exp = env.replay_moves(acts, good)
    for g, e in zip(got, exp):
        np.testing.assert_array_equal(g[~is_bad].cpu().numpy(), e.cpu().numpy())
        assert (g[is_bad] == (-2 if g.dtype == torch.int32 else 0)).all()


def _state(env):
    return [x.cpu().numpy() for x in list(env.export_state().values()) + [env.costs()]]


@pytest.mark.gpu
def test_the_handle_is_untouched_and_each_call_is_one_launch():
    J, M, E = 10, 10, 3
    N = J * M
    d, acts = _random_sequences(J, M, E, 33, True)
    a, b = _env(J, M, E, d, True), _env(J, M, E, d, True)
    lib = libm.lib()
    p = lambda x: C.c_void_p(x.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fresh = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    fresh.load(d["t"], d["p"], d["transT"], d["edge"])
    one = torch.zeros((1, 4), dtype=torch.int32, device=a.device)
    assert lib.mtfjsp_replay_moves(fresh._h, p(one[0, :1]), 1, p(acts.transpose(0, 1).contiguous()), p(one), 1,
                                   None, None, None, st) == E_STATE           # loaded, never reset
    assert b"mtfjsp_replay_moves" in lib.mtfjsp_last_error()
    moves = search.neighbour_moves(acts, torch.as_tensor(d["t"], device=a.device), max_neighbours=64, seed=2)
    for s in range(N):
        if s % 7 == 3:  # after a step: no recorded reset is pending, so the call is its own launch only
            before = _state(a)
            n0 = a.launch_count
            a.replay_moves(acts, moves)
            assert a.launch_count == n0 + 1
            for x, y in zip(before, _state(a)):
                np.testing.assert_array_equal(x, y)
        op, mc = acts[s, :, 0].contiguous(), acts[s, :, 1].contiguous()
        a.step(op, mc)
        b.step(op, mc)
        for k in ("reward5", "scaled4", "done", "invalid"):
            np.testing.assert_array_equal(getattr(a, k).cpu().numpy(), getattr(b, k).cpu().numpy(), err_msg="%d %s" % (s, k))
    for x, y in zip(_state(a), _state(b)):
        np.testing.assert_array_equal(x, y)
    a.check_launch_overlap()
