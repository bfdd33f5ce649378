"""Instance data (SURVEY.md 8 f-4): the stream-compatible generator reproduces the reference's shipped pickles.

The hashes below are SHA-256 prefixes of the four arrays inside ``instance/test_Instance_J6M6E2.pkl`` (seed 3) and
``instance/eval_Instance_J6M6E2.pkl`` (seed 1) of the reference; samples of the pickles themselves (their first 8
instances, same wire format: tests/golden/gen_instance_samples.py) are read back and compared array by array."""
import hashlib
import importlib
import os

import numpy as np
import pytest

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
GOLD = os.path.join(os.path.dirname(__file__), "golden")

SHIPPED = {  # file stem -> (generator seed, sha256[:16] of t, p, transT, edge as int64)
    "test_Instance_J6M6E2": (3, ("92b1284bd57a7ce7", "64aef42a6bedc0a6", "e0506923e8a867ea", "b9dee98b8d49e680")),
    "eval_Instance_J6M6E2": (1, ("0894581e09968da3", "ee1b87e283fe46c1", "d4242bf059821fa2", "b9dee98b8d49e680")),
}


def _h(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


@pytest.mark.parametrize("stem", sorted(SHIPPED))
def test_stream_generator_reproduces_shipped_pickle_hashes(stem):
    seed, want = SHIPPED[stem]
    d = ins.reference_stream_instances(100, 6, 6, 2, seed=seed)
    got = (_h(d["t"]), _h(d["p"]), _h(d["transT"]), _h(d["edge"].astype(np.int64)))
    assert got == want
    assert d["t"].dtype == np.float64 and d["t"].shape == (100, 36, 6) and d["transT"].shape == (100, 6, 6)


@pytest.mark.parametrize("stem", sorted(SHIPPED))
def test_shipped_pickles_equal_generator_output(stem):
    seed, _ = SHIPPED[stem]
    d = ins.reference_stream_instances(100, 6, 6, 2, seed=seed)
    r = ins.load_instances(os.path.join(GOLD, "shipped_%s_first8.pkl" % stem))
    for k in ("t", "p", "transT", "edge"):
        assert len(r[k]) == 8
        np.testing.assert_array_equal(r[k], d[k][:8], err_msg=k)


def test_pickle_wire_format_round_trip(tmp_path):
    """save_instances writes what the reference's loader unpacks: a pickled list of four arrays (generate_...py:286-316)."""
    import pickle

    d = ins.synthetic_instances(0, 5, 10, 10, 3, seed=1003)          # ragged groups 3/3/4, padded with -1
    path = str(tmp_path / "Instance_J10M10E3.pkl")
    ins.save_instances(path, d)
    with open(path, "rb") as f:
        t, p, tt, edge = pickle.load(f)                              # the reference's own unpacking
    assert t.dtype == np.float64 and edge.dtype == np.int64 and edge.shape == (5, 3, 4)
    back = ins.load_instances(path)
    for k in d:
        np.testing.assert_array_equal(back[k], d[k], err_msg=k)


def test_synthetic_slices_agree_with_whole_batch():
    whole = ins.synthetic_instances(0, 3000, 6, 6, 2, seed=7)
    part = ins.synthetic_instances(1500, 700, 6, 6, 2, seed=7)
    for k in whole:
        np.testing.assert_array_equal(whole[k][1500:2200], part[k])
    t, p = whole["t"], whole["p"]
    assert ((t >= 0).sum(-1) >= 1).all() and ((t < 0) == (p < 0)).all()   # at least one feasible machine per op
    tt = whole["transT"]
    assert (tt == np.transpose(tt, (0, 2, 1))).all() and (np.diagonal(tt, axis1=1, axis2=2) == 0).all()


@pytest.mark.gpu
def test_device_generator_draws_the_reference_distributions():
    """mtfjsp_generate_instances (SURVEY.md 8 f-4): ranges and structure of generate_allsize_mofjsp_dataset.py:161-273,
    slices equal the whole batch, and the env steps on what it produced."""
    torch = pytest.importorskip("torch")
    J, M, E, B = 10, 10, 3, 4096
    d = ins.device_instances(0, B, J, M, E, seed=11)
    t, p, tt, edge = (d[k].cpu().numpy() for k in ("t", "p", "transT", "edge"))
    assert ((t < 0) == (p < 0)).all() and ((t >= 0).sum(-1) >= 1).all()
    at, ap = np.abs(t), np.abs(p)
    assert at.min() >= 0.8 * 1 and at.max() <= 1.2 * 99 and ap.min() >= 0.8 and ap.max() <= 1.2 * 20
    assert 49.0 < at.mean() < 51.0 and 10.2 < ap.mean() < 10.8                    # E[U(1,99)] = 50, E[U(1,20)] = 10.5
    frac_neg = (t < 0).mean()
    assert abs(frac_neg - (M - 1) / (2 * M)) < 0.01                                # k ~ randint(0, M): mean (M-1)/2 of M
    k = (t < 0).sum(-1)
    assert k.min() == 0 and k.max() == M - 1 and len(np.unique(k)) == M
    assert (tt == np.transpose(tt, (0, 2, 1))).all() and (np.diagonal(tt, axis1=1, axis2=2) == 0).all()
    np.testing.assert_array_equal(edge[0], ins.edge_groups(M, E))
    gid = ins.edge_of_machine(edge[0], M)
    dist = np.abs(gid[:, None] - gid[None, :])
    off = ~np.eye(M, dtype=bool)
    lo = np.where(dist == 0, 1.0, 10.0 * dist); hi = np.where(dist == 0, 10.0, 20.0 * dist)
    assert (tt[:, off] >= lo[off]).all() and (tt[:, off] <= hi[off]).all()
    part = ins.device_instances(1000, 300, J, M, E, seed=11)
    for kname in ("t", "p", "transT", "edge"):
        assert torch.equal(part[kname], d[kname][1000:1300])
    other = ins.device_instances(0, 64, J, M, E, seed=12)
    assert not torch.equal(other["t"], d["t"][:64])
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 11))
    for _ in range(J * M):
        env.random_step(seed=3)
    assert bool(env.done.all()) and not bool(env.invalid.any())
