"""The reference's idle-time lookahead rule (tester/pdrs.py:465-540, LWKR_IT_o_jointActor) against its own recorded run
(tests/golden/lookahead_golden.npz): a CPU restatement on the oracle env that replays the chosen prefix and steps each
candidate, as the reference does, reproduces every recorded it_temp bit for bit and, following the recorded choices, the
final costs; the device rule's decision (rules.lookahead_choice) takes the reference's choice wherever it is unique and
the lowest job index where the reference drew among ties."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

GOLD = os.path.join(os.path.dirname(__file__), "golden", "lookahead_golden.npz")
NAME = {"min": "LWKR_IT", "max": "MWKR_IT"}


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def oracle():
    mod = importlib.import_module("oracle.mtfjsp_oracle")
    mod.build()
    return mod


def _instance(g, r):
    i = int(g["run_inst"][r])
    if int(g["run_J"][r]) == 6:
        return g["t"][i], g["p"][i], g["transT"][i], g["edge"][i]
    return g["t10"][i], g["p10"][i], g["transT10"][i], g["edge10"][i]


def _oracle_env(oracle, g, r, B):
    J, M = int(g["run_J"][r]), int(g["run_M"][r])
    t, p, tt, e = _instance(g, r)
    env = oracle.OracleEnv(B, J, M, 2, left_shift=False)
    env.load(np.repeat(t[None], B, 0), np.repeat(p[None], B, 0), np.repeat(tt[None], B, 0), np.repeat(e[None], B, 0))
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (B, 1)))
    return env


def _chosen_ops(g, r):
    J, M = int(g["run_J"][r]), int(g["run_M"][r])
    nx = [0] * J
    ops = []
    for s in range(J * M):
        j = int(g["chosen"][r, s])
        ops.append(j * M + nx[j])
        nx[j] += 1
    return np.array(ops)


def _runs(g):
    return range(len(g["run_J"]))


def test_replay_restatement_reproduces_every_it_temp(gold, oracle):
    """Per decision: one oracle env per candidate job replays the chosen prefix, then steps its candidate op on the
    listed machine; its r_idle is the recorded it_temp, bit for bit."""
    g = gold
    for r in _runs(g):
        J, M = int(g["run_J"][r]), int(g["run_M"][r])
        ml = g["mlist"][r].astype(np.int32)
        ops = _chosen_ops(g, r)
        for s in range(J * M):
            jobs = g["cand"][r, s][g["cand"][r, s] >= 0].astype(np.int32)
            env = _oracle_env(oracle, g, r, len(jobs))
            for a in ops[:s]:
                env.step(np.full(len(jobs), a), np.full(len(jobs), ml[a]))
            nx = np.array([np.sum(ops[:s] // M == j) for j in jobs])
            cop = jobs * M + nx
            r5, _, _, inv = env.step(cop, ml[cop])
            assert not inv.any()
            np.testing.assert_array_equal(r5[:, 2], g["it"][r, s, :len(jobs)], err_msg="run %d step %d" % (r, s))


def test_recorded_choices_reproduce_the_final_costs(gold, oracle):
    g = gold
    for r in _runs(g):
        J, M = int(g["run_J"][r]), int(g["run_M"][r])
        ml = g["mlist"][r].astype(np.int32)
        env = _oracle_env(oracle, g, r, 1)
        for a in _chosen_ops(g, r):
            _, _, done, inv = env.step(np.array([a]), np.array([ml[a]]))
            assert not inv.any()
        assert done.all()
        np.testing.assert_array_equal(env.costs()[0], g["final4"][r], err_msg="run %d" % r)


def test_lowest_index_tie_break_on_the_recorded_decisions(gold):
    """rules.lookahead_choice on every recorded decision: the reference's job where its best it_temp is unique, the
    lowest tied job where the reference drew with random.choice (the fixture has such steps)."""
    rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")
    g = gold
    tied = 0
    for r in _runs(g):
        J, M = int(g["run_J"][r]), int(g["run_M"][r])
        kind = str(g["run_type"][r])
        ridle = torch.zeros((J * M, J), dtype=torch.float64)
        inv = torch.ones((J * M, J), dtype=torch.uint8)
        for s in range(J * M):
            jobs = g["cand"][r, s][g["cand"][r, s] >= 0]
            ridle[s, jobs] = torch.from_numpy(g["it"][r, s, :len(jobs)])
            inv[s, jobs] = 0
        got = rules.lookahead_choice(NAME[kind], ridle, inv)[:, 0].numpy()
        for s in range(J * M):
            jobs = g["cand"][r, s][g["cand"][r, s] >= 0]
            it = g["it"][r, s, :len(jobs)]
            best = it.max() if kind == "min" else it.min()
            ties = jobs[it == best]
            assert got[s] == ties.min(), (r, s)
            if len(ties) == 1:
                assert got[s] == g["chosen"][r, s], (r, s)
            else:
                tied += 1
                assert g["chosen"][r, s] in ties, (r, s)
    assert tied > 0
