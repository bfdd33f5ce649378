"""Golden call sequences of the reference's single-env class for tests/test_single_env.py (single_env_golden.npz).

Run where a checkout of the reference project is available (no GPU needed):

    MTFJSP_REFERENCE_ROOT=<reference checkout> python tests/golden/gen_single_env_golden.py

Three groups, each recorded from the reference class (digests: oracle/single_env_trace.py):
  step/<cfg>/*  reset and step returns, valid-action masks, node attributes, machine routes and final costs along seeded
                random actions, both reward-weight draws, two instances per configuration;
  pdr/*         the unmodified dispatching-rule rollout tester/pdrs.py:611-839 for four rules on the first 12 shipped test
                instances (its actions are pdr_golden.npz's op / machine orders): what each call returned;
  validate/*    the unmodified validation loop trainer/validate.py:60-297 with the reference networks and the shipped
                checkpoint, on the CPU, on the first 10 shipped test instances: its actions, what each call returned, the
                final costs and the objective it reports.
"""
import contextlib
import io
import os
import random
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import importlib  # noqa: E402

from oracle import ref_harness as rh  # noqa: E402
from oracle import single_env_trace as tr  # noqa: E402

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")


def gen_steps(ref, out):
    for cfg in tr.STEP_CFGS:
        J, M, E, ls, seed = cfg
        N = J * M
        key = "step/%s/" % tr.cfg_key(cfg)
        d = ins.reference_stream_instances(4, J, M, E, seed=3) if (J, M) == (6, 6) else ins.synthetic_instances(0, 4, J, M, E, seed)
        args = rh.make_args(J, M, E, 1)
        rng = np.random.default_rng(seed)
        acts = np.zeros((2, 2, N, 2), dtype=np.int16)
        weights = np.zeros((2, 2, 3))
        resets = np.zeros((2, 2, 9), dtype=np.uint64)
        steps = np.zeros((2, 2, N, 14), dtype=np.uint64)
        state = np.zeros((2, 2, N, 3), dtype=np.uint64)     # valid-action mask before the step, nodes and routes after it
        final = np.zeros((2, 2, 4))
        for i in range(2):
            t, p, tt = d["t"][i], d["p"][i], d["transT"][i]
            env = tr.make_env(ref.Env, t, p, tt, args, ls)
            for k, kind in enumerate(("eval", "01")):
                random.seed(11 + i)
                resets[i, k] = tr.tuple_digests(env.reset(Random_weight_type=kind))
                weights[i, k] = env.reward_random_weight
                nxt = np.zeros(J, dtype=int)
                for s in range(N):
                    mask = tr.digest(env.valid_action_mask())
                    j = rng.choice(np.nonzero(nxt < M)[0])
                    op = j * M + nxt[j]
                    nxt[j] += 1
                    feas = np.nonzero(t[op] >= 0)[0]
                    m = feas[0] if rng.random() < 0.4 else rng.choice(feas)   # lowest index: same-machine chains
                    acts[i, k, s] = op, m
                    sa = tr.step_quiet(env, (op, m))
                    steps[i, k, s] = tr.tuple_digests(sa)
                    state[i, k, s] = mask, tr.nodes_digest(env, N), tr.routes_digest(env, M)
                assert sa[2] is True or sa[2] == True  # noqa: E712
                final[i, k] = [env.makespan_previous_step, env.total_e1_previous_step, env.trans_t_previous_step,
                               env.idle_t_previous_step]
        out.update({key + "actions": acts, key + "weights": weights, key + "reset": resets, key + "step": steps,
                    key + "state": state, key + "final": final})


def recording_class(ref, log, nodes=False):
    class Recording(ref.Env):
        def reset(self, *a, **kw):
            r = super().reset(*a, **kw)
            log.append(("reset", None, tr.combined_digest(r), None))
            return r

        def step(self, joint_action):
            r = super().step(joint_action)
            nd = tr.nodes_digest(self, self.total_tasks_without_dummies) if nodes else None
            log.append(("step", (int(joint_action[0]), int(joint_action[1])), tr.combined_digest(r), nd))
            return r

    return Recording


def split_episode(log, N):
    """reset("eval"), N steps, the trailing reset() (its weights come from python's global `random`: not kept)."""
    assert [e[0] for e in log] == ["reset"] + ["step"] * N + ["reset"], [e[0] for e in log]
    steps = log[1:N + 1]
    return (log[0][2], np.array([e[1] for e in steps], dtype=np.int16), np.array([e[2] for e in steps], dtype=np.uint64),
            np.array([e[3] for e in steps], dtype=np.uint64) if steps[0][3] is not None else None)


def gen_pdr(ref, out):
    if "trainer.fig_kpi" not in sys.modules:
        fk = types.ModuleType("trainer.fig_kpi")
        fk.result_box_plot = lambda *a, **k: None
        fk.get_GPU_usage = lambda *a, **k: None
        sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from tester import pdrs
    g = np.load(os.path.join(HERE, "pdr_golden.npz"))
    ds = types.SimpleNamespace(t=g["t"], p=g["p"], transT=g["transT"], edge=g["edge"])
    args = rh.make_args(6, 6, 2, 1)
    log = []
    pdrs.DisjunctiveGraphJspEnv_singleStep = recording_class(ref, log)
    resets = np.zeros((len(tr.PDR_ROWS), tr.PDR_INSTANCES), dtype=np.uint64)
    steps = np.zeros((len(tr.PDR_ROWS), tr.PDR_INSTANCES, 36), dtype=np.uint64)
    for r, ((o_rule, m_rule), row) in enumerate(tr.PDR_ROWS.items()):
        for i in range(tr.PDR_INSTANCES):
            log.clear()
            with contextlib.redirect_stdout(io.StringIO()):
                _, _, real4 = pdrs.run_Rules_jointActions_withMinus_1217(args, o_rule, m_rule, ds, i, None, None)
            np.testing.assert_array_equal(np.array(real4), g["gold"][row, i])
            resets[r, i], acts, steps[r, i], _ = split_episode(log, 36)
            np.testing.assert_array_equal(acts[:, 0], g["ops"][row, i])
            np.testing.assert_array_equal(acts[:, 1], g["mch"][row, i])
    out.update({"pdr/reset": resets, "pdr/step": steps})


def gen_validate(ref, out):
    import torch

    cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda t, *a, **k: t   # the reference moves a few masks with .cuda(); everything runs on the CPU here
    try:
        ppo, args = rh.make_reference_ppo(6, 6, "cpu")
        with contextlib.redirect_stdout(io.StringIO()):
            from trainer import validate
    except BaseException:
        torch.Tensor.cuda = cuda
        raise
    g = np.load(os.path.join(HERE, "pdr_golden.npz"))   # the 100 shipped test instances
    ds = types.SimpleNamespace(t=g["t"], p=g["p"], transT=g["transT"], edge=g["edge"])
    log = []
    validate.DisjunctiveGraphJspEnv_singleStep = recording_class(ref, log, nodes=True)
    n = tr.VALIDATE_INSTANCES
    resets = np.zeros(n, dtype=np.uint64)
    acts = np.zeros((n, 36, 2), dtype=np.int16)
    steps = np.zeros((n, 36), dtype=np.uint64)
    nodes = np.zeros((n, 36), dtype=np.uint64)
    final = np.zeros((n, 5))
    try:
        for i in range(n):
            log.clear()
            random.seed(i)
            torch.manual_seed(0)
            with contextlib.redirect_stdout(io.StringIO()):
                _, final4, obj = validate.validate_cost_gcn_jointActor_GAT(ppo, False, ds, i, "random", greedy=True, args=args)
            final[i] = list(final4) + [obj]
            resets[i], acts[i], steps[i], nodes[i] = split_episode(log, 36)
    finally:
        torch.Tensor.cuda = cuda
    out.update({"validate/reset": resets, "validate/actions": acts, "validate/step": steps, "validate/nodes": nodes,
                "validate/final": final})


def main():
    ref = rh.load_reference()
    out = {}
    gen_steps(ref, out)
    gen_pdr(ref, out)
    gen_validate(ref, out)
    np.savez_compressed(os.path.join(HERE, "single_env_golden.npz"), **out)
    print("single_env_golden.npz:", ", ".join("%s %s" % (k, v.shape) for k, v in out.items()))


if __name__ == "__main__":
    main()
