"""Generates tests/golden/lookahead_golden.npz from the real reference (a checkout named by MTFJSP_REFERENCE_ROOT, read
through oracle/ref_harness.py): the reference's own idle-time
lookahead rule FJSP_Rules.LWKR_IT_o_jointActor (tester/pdrs.py:465-540), run the way run_Rules_jointActions_withMinus_1217
(tester/pdrs.py:611-680) builds its env: perform_left_shift_if_possible=False, reset(Random_weight_type="eval"), the
machine list (SPT_m / SEC_m) computed first.

    MTFJSP_REFERENCE_ROOT=<reference checkout> python tests/golden/gen_lookahead_golden.py

Runs: type "min" and "max" x SPT and SEC on the 8 instances of shipped_test_Instance_J6M6E2_first8.pkl, and "min" + SPT
on the first J10M10E2 instance of the reference generator stream (seed 3).  python's random is seeded per run (the rule
breaks ties with random.choice).  Per run and step it records the candidate jobs (the rule's index_list: jobs with an
unscheduled op, ascending), their it_temp values (r_idle of stepping the candidate op on its listed machine after
replaying the chosen prefix) and the chosen job; per run the machine list and the final (makespan, processing energy / N,
transport time, idle time) of the chosen sequence.

Layout (R runs, N_max = 100 steps, J_max = 10 jobs; shorter runs padded with -1 / NaN):
  run_J, run_M [R], run_type [R] ("min" / "max"), run_mrule [R] ("SPT" / "SEC"), run_inst [R] (index into its set),
  cand [R,N_max,J_max] int8 (-1 padded), it [R,N_max,J_max] f64 (NaN padded), chosen [R,N_max] int8 (job),
  mlist [R,100] int8 (machine of every op, -1 padded), final4 [R,4] f64,
  j6 instances t, p, transT, edge; j10 instance t10, p10, transT10, edge10.
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

from oracle import ref_harness as rh  # noqa: E402

import importlib.util  # noqa: E402

_spec = importlib.util.spec_from_file_location("instances", os.path.join(ROOT, "e2e-mappo-for-mt-fjsp_b200", "instances.py"))
ins = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(ins)

N_MAX, J_MAX = 100, 10


class _Recorder:
    """Wraps the reference env: the r_idle of the last step before each reset() is one candidate's it_temp entry."""

    def __init__(self, env):
        self.env, self.last, self.its = env, None, []

    def step(self, *a, **k):
        out = self.env.step(*a, **k)
        self.last = out[5]
        return out

    def reset(self, *a, **k):
        if self.last is not None:
            self.its.append(float(self.last))
            self.last = None
        return self.env.reset(*a, **k)

    def __getattr__(self, name):
        return getattr(self.env, name)


def run(pdrs, ns, J, M, E, t, p, tt, kind, mrule, seed):
    args = rh.make_args(J, M, E, 1)
    rules = pdrs.FJSP_Rules(J, M)
    mlist = rules.SPT_m(t) if mrule == "SPT" else rules.SEC_m(t, p)
    env = ns.Env(jps_instance=np.array([t, p]), reward_function_parameters=args["reward_scaling"],
                 default_visualisations=["gantt_console", "graph_console"], reward_function="wrk", ability_tr_mm=tt,
                 perform_left_shift_if_possible=False, configs=args)
    env.reset(Random_weight_type="eval")
    rec = _Recorder(env)
    random.seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        chosen = rules.LWKR_IT_o_jointActor(rec, kind, mlist)
    ops = [c - 1 for c in chosen]
    N = J * M
    assert sorted(ops) == list(range(N))
    cand = np.full((N_MAX, J_MAX), -1, dtype=np.int8)
    it = np.full((N_MAX, J_MAX), np.nan)
    pick = np.full(N_MAX, -1, dtype=np.int8)
    nx = [0] * J
    k = 0
    for s, a in enumerate(ops):
        jobs = [j for j in range(J) if nx[j] < M]
        cand[s, :len(jobs)] = jobs
        it[s, :len(jobs)] = rec.its[k:k + len(jobs)]
        k += len(jobs)
        pick[s] = a // M
        assert a == (a // M) * M + nx[a // M]
        nx[a // M] += 1
    assert k == len(rec.its)
    # the chosen sequence, as run_Rules_jointActions_withMinus_1217 rolls it out (the rule left the env reset)
    with contextlib.redirect_stdout(io.StringIO()):
        for a in ops:
            done = env.step(joint_action=[a, mlist[a]])[2]
    assert done
    final4 = [env.makespan_previous_step, env.total_e1_previous_step / N, env.trans_t_previous_step,
              env.idle_t_previous_step]
    ml = np.full(N_MAX, -1, dtype=np.int8)
    ml[:N] = mlist
    return cand, it, pick, ml, np.array(final4, dtype=np.float64)


def main():
    ns = rh.load_reference()
    fk = types.ModuleType("trainer.fig_kpi")
    fk.result_box_plot = lambda *a, **k: None
    sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from tester import pdrs
    d6 = ins.load_instances(os.path.join(HERE, "shipped_test_Instance_J6M6E2_first8.pkl"))
    d10 = ins.reference_stream_instances(1, 10, 10, 2, seed=3)
    runs = []
    for kind in ("min", "max"):
        for mrule in ("SPT", "SEC"):
            for i in range(8):
                runs.append((6, 6, kind, mrule, i))
    runs.append((10, 10, "min", "SPT", 0))
    out = {k: [] for k in ("cand", "it", "chosen", "mlist", "final4")}
    for r, (J, M, kind, mrule, i) in enumerate(runs):
        d = d6 if J == 6 else d10
        res = run(pdrs, ns, J, M, 2, d["t"][i], d["p"][i], d["transT"][i], kind, mrule, seed=1000 + r)
        for k, v in zip(("cand", "it", "chosen", "mlist", "final4"), res):
            out[k].append(v)
        print("run %d J%dM%d %s+%s inst %d: final4 %s" % (r, J, M, kind, mrule, i, res[4]), flush=True)
    np.savez_compressed(
        os.path.join(HERE, "lookahead_golden.npz"),
        run_J=np.array([r[0] for r in runs]), run_M=np.array([r[1] for r in runs]),
        run_type=np.array([r[2] for r in runs]), run_mrule=np.array([r[3] for r in runs]),
        run_inst=np.array([r[4] for r in runs]),
        **{k: np.stack(v) for k, v in out.items()},
        t=d6["t"], p=d6["p"], transT=d6["transT"], edge=np.asarray(d6["edge"]),
        t10=d10["t"][:1], p10=d10["p"][:1], transT10=d10["transT"][:1], edge10=np.asarray(d10["edge"])[:1])


if __name__ == "__main__":
    main()
