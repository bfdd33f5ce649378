"""The single-env class (reference: graph-jsp-env/.../disjunctive_graph_jsp_env_singlestep.py:97-130 ctor,
1183-1245 reset -> 9-tuple, 716-974 step -> 14-tuple) against the UNMODIFIED reference, on the GPU box.

What the reference class returned is stored in tests/golden/single_env_golden.npz (tests/golden/gen_single_env_golden.py;
digests of canonical forms, oracle/single_env_trace.py), so these tests need nothing outside the repository.  Three layers:
  1. every element of the reset 9-tuple and step 14-tuple, the node attributes, machine routes, final-cost attributes
     and the valid-action mask, step by step against the reference class on the same actions (both left-shift modes);
  2. the calls the unmodified dispatching-rule rollout tester/pdrs.py:611-839 makes, replayed on OUR class: every return
     as the reference class gave it, and the shipped result CSV rows 0 / 1 / 4 / 11 bit for bit;
  3. the calls the unmodified validation loop trainer/validate.py:60-297 makes with the reference's own networks and the
     shipped checkpoint, replayed on OUR class: every return, node attribute, final cost and the objective as with the
     reference class, bit for bit.
"""
import importlib
import os
import random

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import ref_harness as rh  # noqa: E402
from oracle import single_env_trace as tr  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
eq = np.testing.assert_array_equal


def _mine():
    return importlib.import_module("e2e-mappo-for-mt-fjsp_b200.single_env").DisjunctiveGraphJspEnv_singleStep


def _golden():
    return np.load(os.path.join(GOLD, "single_env_golden.npz"))


def _same(got, want, what):
    """Digests of what our class returned against the reference class's."""
    got, want = np.atleast_1d(np.asarray(got, dtype=np.uint64)), np.atleast_1d(want)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, "%s: element(s) %s differ from the reference" % (what, bad.tolist())


@pytest.mark.parametrize("cfg", tr.STEP_CFGS)
def test_tuples_and_attributes_match_the_reference_class_step_by_step(cfg):
    J, M, E, ls, seed = cfg
    N = J * M
    g, key = _golden(), "step/%s/" % tr.cfg_key(cfg)
    acts, resets, steps, state, final = (g[key + k] for k in ("actions", "reset", "step", "state", "final"))
    d = ins.reference_stream_instances(4, J, M, E, seed=3) if (J, M) == (6, 6) else ins.synthetic_instances(0, 4, J, M, E, seed)
    args = rh.make_args(J, M, E, 1)
    for i in range(2):
        t, p, tt = d["t"][i], d["p"][i], d["transT"][i]
        env = tr.make_env(_mine(), t, p, tt, args, ls)
        for k, kind in enumerate(("eval", "01")):
            random.seed(11 + i)
            rb = env.reset(Random_weight_type=kind)
            assert len(rb) == 9
            _same(tr.tuple_digests(rb), resets[i, k], "reset")
            eq(env.reward_random_weight, g[key + "weights"][i, k])
            for s in range(N):
                _same(tr.digest(env.valid_action_mask()), state[i, k, s, 0], "valid_action_mask s=%d" % s)
                sb = tr.step_quiet(env, acts[i, k, s])
                assert len(sb) == 14
                _same(tr.tuple_digests(sb), steps[i, k, s], "step s=%d" % s)
                _same(tr.nodes_digest(env, N), state[i, k, s, 1], "node attributes s=%d" % s)
                _same(tr.routes_digest(env, M), state[i, k, s, 2], "machine routes s=%d" % s)
            got = [env.makespan_previous_step, env.total_e1_previous_step, env.trans_t_previous_step, env.idle_t_previous_step]
            eq(np.array(got), final[i, k])
            assert sb[2] is True
        assert "M0" in env.render(mode="text")
        env.close()


def test_unmodified_pdr_rollout_reproduces_shipped_csv_rows_on_our_class():
    g, pdr = _golden(), np.load(os.path.join(GOLD, "pdr_golden.npz"))
    args = rh.make_args(6, 6, 2, 1)
    for r, ((o_rule, m_rule), row) in enumerate(tr.PDR_ROWS.items()):
        for i in range(tr.PDR_INSTANCES):
            what = "rule %s instance %d" % ((o_rule, m_rule), i)
            env = tr.make_env(_mine(), pdr["t"][i], pdr["p"][i], pdr["transT"][i], args, False)
            _same(tr.combined_digest(env.reset(Random_weight_type="eval")), g["pdr/reset"][r, i], what + " reset")
            for s in range(36):
                out = tr.step_quiet(env, (pdr["ops"][row, i, s], pdr["mch"][row, i, s]))
                _same(tr.combined_digest(out), g["pdr/step"][r, i, s], what + " step %d" % s)
            assert out[2]
            eq(np.array(tr.final_costs(env, 36)), pdr["gold"][row, i], err_msg=what)
            env.reset()
            env.close()


def test_unmodified_validation_loop_with_shipped_checkpoint_on_our_class():
    g, pdr = _golden(), np.load(os.path.join(GOLD, "pdr_golden.npz"))   # the 100 shipped test instances
    args = rh.default_model_args(6, 6)
    res = []
    for i in range(tr.VALIDATE_INSTANCES):
        env = tr.make_env(_mine(), pdr["t"][i], pdr["p"][i], pdr["transT"][i], args, True)
        _same(tr.combined_digest(env.reset(Random_weight_type="eval")), g["validate/reset"][i], "instance %d reset" % i)
        for s in range(36):
            out = tr.step_quiet(env, g["validate/actions"][i, s])
            _same(tr.combined_digest(out), g["validate/step"][i, s], "instance %d step %d" % (i, s))
            _same(tr.nodes_digest(env, 36), g["validate/nodes"][i, s], "instance %d node attributes after step %d" % (i, s))
        assert out[2]
        mk, pt, transT, idleT = tr.final_costs(env, 36)
        res.append([mk, pt, transT, idleT, args["weight_mk"] * mk + args["weight_ec"] * (pt + idleT) + args["weight_tt"] * transT])
        random.seed(i)
        env.reset()
        env.close()
    res = np.array(res)
    eq(res, g["validate/final"])
    assert np.isfinite(res).all() and (res[:, 0] > 0).all()
