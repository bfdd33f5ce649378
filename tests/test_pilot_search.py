"""search.pilot_search: the pilot method on the device episode completion.  On the 100 shipped J6M6 test instances
(tests/golden/pdr_golden.npz) with FIFO+SPT and MWKR_T+SPT as the base under both candidate sets: never worse than the
rule's shipped row, a history that never increases and ends at the returned objective, returned sequences that replay
to the returned costs, and one instance alone giving the result it gets in the batch.  The random base: deterministic
for a seed, its objective the history's minimum, its sequences replaying to its costs."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
search = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.search")
validate = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")

PDR = os.path.join(os.path.dirname(__file__), "golden", "pdr_golden.npz")


def _instances(sl=slice(None)):
    g = np.load(PDR)
    return {k: g[k][sl] for k in ("t", "p", "transT", "edge")}, g


def _replay(inst, actions, left_shift=False):
    S = inst["t"].shape[0]
    env = envm.BatchedMTFJSPEnv(S, 6, 6, 2, left_shift=left_shift, obs_dtype=torch.float32)
    env.load(inst["t"], inst["p"], inst["transT"], inst["edge"])
    env.scaler_init()
    env.reset(np.tile([0.4, 0.4, 0.2], (S, 1)))
    f4, _, fi = env.replay(torch.as_tensor(actions, device=env.device))
    out = f4.cpu().numpy(), fi.cpu().numpy()
    env.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("candidates", ["all", "rule"])
@pytest.mark.parametrize("rule", ["FIFO+SPT", "MWKR_T+SPT"])
def test_priority_pilot_improves_on_its_rule(rule, candidates):
    inst, g = _instances()
    row = [str(x) for x in g["rule_names"]].index(rule)
    rule_obj = validate._objective(g["gold"][row], (0.4, 0.4, 0.2))
    out = search.pilot_search(inst, base=tuple(rule.split("+")), candidates=candidates)
    h = out["history"]
    assert h.shape == (37, 100) and out["actions"].shape == (36, 100, 2)
    np.testing.assert_array_equal(h[0], rule_obj)
    np.testing.assert_array_equal(out["base_objective"], rule_obj)
    assert (np.diff(h, axis=0) <= 0).all()
    np.testing.assert_array_equal(out["objective"], h[-1])
    np.testing.assert_array_equal(out["objective"], h.min(0))
    assert (out["objective"] <= rule_obj).all()
    f4, fi = _replay(inst, out["actions"])
    assert (fi == -1).all()
    np.testing.assert_array_equal(f4, out["final4"])
    np.testing.assert_array_equal(validate._objective(f4, (0.4, 0.4, 0.2)), out["objective"])
    one, _ = _instances(slice(37, 38))
    alone = search.pilot_search(one, base=tuple(rule.split("+")), candidates=candidates, max_candidates=7)
    for k in ("actions", "final4", "objective", "history"):
        np.testing.assert_array_equal(alone[k], out[k][..., 37:38, :] if k in ("actions",) else
                                      (out[k][37:38] if k in ("final4", "objective") else out[k][:, 37:38]), err_msg=k)


@pytest.mark.gpu
def test_random_pilot_is_deterministic_and_replays():
    inst, _ = _instances(slice(0, 12))
    a = search.pilot_search(inst, base="random", samples=2, seed=5)
    b = search.pilot_search(inst, base="random", samples=2, seed=5)
    for k in ("actions", "final4", "objective", "history"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    np.testing.assert_array_equal(a["objective"], a["history"].min(0))
    f4, fi = _replay(inst, a["actions"])
    assert (fi == -1).all()
    np.testing.assert_array_equal(f4, a["final4"])
    assert a["completions"] == 12 * 2 + 36 * 12 * 36 * 2
    with pytest.raises(ValueError):
        search.pilot_search(inst, base="random", candidates="rule")
