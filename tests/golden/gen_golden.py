"""Generates the golden fixtures in this directory from the REAL reference (/root/reference).

Run in the build container only (the reference tree is not present on the GPU box):

    python tests/golden/gen_golden.py

Outputs
  pdr_golden.npz     the reference's shipped result rows (results/test_results/Real_{MK,PT,TT,IT}_J6_M6_E2_Seed3_Weight442.csv,
                     rows FIFO/LWKR_T/LWKR_PT/MWKR_T/MWKR_PT x SPT/SEC = CSV rows 0,1,4..11) for the 100 shipped test
                     instances, the op / machine orders the reference's own rule code (tester/pdrs.py) produces for
                     them, and the test instances themselves.  Before writing, every row is re-run through the
                     unmodified reference rollout (tester/pdrs.py:611-839) and must reproduce the CSV exactly.
  replay_*.npz       per-step dumps of the reference ``Parallel_env`` (trainer/parallel_env.py) + job-mask rule
                     (algorithm/ppo_algorithm.py:202-317) on seeded instances and recorded random actions.
"""
import csv
import io
import contextlib
import os
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

REF = rh.REF_ROOT
CSV_ROWS = [0, 1, 4, 5, 6, 7, 8, 9, 10, 11]
RULES = [(0, 0), (0, 1), (2, 0), (2, 1), (3, 0), (3, 1), (4, 0), (4, 1), (5, 0), (5, 1)]  # (o_rule, m_rule), test_all.py:484-503
RULE_NAMES = ["FIFO+SPT", "FIFO+SEC", "LWKR_T+SPT", "LWKR_T+SEC", "LWKR_PT+SPT", "LWKR_PT+SEC",
              "MWKR_T+SPT", "MWKR_T+SEC", "MWKR_PT+SPT", "MWKR_PT+SEC"]


def gen_pdr():
    rh.load_reference()
    fk = types.ModuleType("trainer.fig_kpi")
    fk.result_box_plot = lambda *a, **k: None
    sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from tester import pdrs
    data = ins.reference_stream_instances(100, 6, 6, 2, seed=3)
    ds = types.SimpleNamespace(t=data["t"], p=data["p"], transT=data["transT"], edge=data["edge"])
    gold = np.zeros((len(CSV_ROWS), 100, 4))
    for k, name in enumerate(("MK", "PT", "TT", "IT")):  # untilNow order = [mk, pt, transT, idleT]
        rows = list(csv.reader(open(os.path.join(REF, "results/test_results/Real_%s_J6_M6_E2_Seed3_Weight442.csv" % name))))
        for r, cr in enumerate(CSV_ROWS):
            gold[r, :, k] = [float(x) for x in rows[cr][:100]]
    args = rh.make_args(6, 6, 2, 1)
    rules = pdrs.FJSP_Rules(6, 6)
    ops = np.zeros((len(RULES), 100, 36), dtype=np.int16)
    mch = np.zeros((len(RULES), 100, 36), dtype=np.int16)
    worst = 0.0
    for r, (o_rule, m_rule) in enumerate(RULES):
        for i in range(100):
            t, p = data["t"][i], data["p"][i]
            if o_rule == 0:
                ol = rules.FIFO_o()
            elif o_rule == 2:
                ol = rules.LWKR_T_o_jointActor(t, "mean", rule_type="least")
            elif o_rule == 3:
                ol = rules.LWKR_PT_o_jointActor(t, p, "mean", rule_type="least")
            elif o_rule == 4:
                ol = rules.LWKR_T_o_jointActor(t, "mean", rule_type="most")
            else:
                ol = rules.LWKR_PT_o_jointActor(t, p, "mean", rule_type="most")
            ml = rules.SPT_m(t) if m_rule == 0 else rules.SEC_m(t, p)
            ops[r, i] = np.array(ol) - 1
            mch[r, i] = [ml[o - 1] for o in ol]
            with contextlib.redirect_stdout(io.StringIO()):
                _, _, real4 = pdrs.run_Rules_jointActions_withMinus_1217(args, o_rule, m_rule, ds, i, None, None)
            err = np.max(np.abs(np.array(real4) - gold[r, i]) / np.abs(gold[r, i]))
            worst = max(worst, err)
            assert err == 0.0, (RULE_NAMES[r], i, real4, gold[r, i])
    print("pdr rows reproduce the shipped CSVs, max rel err", worst)
    np.savez_compressed(os.path.join(HERE, "pdr_golden.npz"), gold=gold, ops=ops, mch=mch, t=data["t"], p=data["p"],
                        transT=data["transT"], edge=data["edge"], rule_names=np.array(RULE_NAMES), csv_rows=np.array(CSV_ROWS))


REPLAYS = [
    # name, J, M, E, B, left_shift, mask_mode, machine policy, duration scale, episodes, seed
    ("j6m6_ls_esa", 6, 6, 2, 4, True, 1, "random", 1.0, 2, 101),
    ("j6m6_ls_fin_mixed_tiny", 6, 6, 2, 4, True, 0, "mixed", 0.02, 1, 102),
    ("j6m6_nols_fin_lowest", 6, 6, 2, 2, False, 0, "lowest", 1.0, 1, 103),
    ("j6m6_ls_fin_lowest", 6, 6, 2, 4, True, 0, "lowest", 1.0, 1, 104),
    ("j3m4_ls_fin_mixed", 3, 4, 2, 4, True, 0, "mixed", 1.0, 2, 105),
    ("j10m10e3_ls_esa_mixed", 10, 10, 3, 2, True, 1, "mixed", 1.0, 1, 106),
    ("j10m10e3_ls_fin_mixed", 10, 10, 3, 1, True, 0, "mixed", 1.0, 1, 107),
    # two more sizes of the reference generator's list; J15M10 has N = 150 > 128: numpy's pairwise summation splits
    ("j20m6e3_ls_esa_mixed", 20, 6, 3, 2, True, 1, "mixed", 1.0, 1, 108),
    ("j15m10e2_ls_fin_mixed", 15, 10, 2, 1, True, 0, "mixed", 1.0, 1, 109),
    # BASELINE.json configs[3]: N = 600 (5 numpy pairwise leaves, the 32-lane kernel with aliased scratch).  One env, one
    # episode = 600 reference steps at ~0.3 s; the bulky dumps are kept at SPARSE_STEPS only
    ("j30m20e5_ls_esa_mixed", 30, 20, 5, 1, True, 1, "mixed", 1.0, 1, 110),
    # the edges of the size range: M = 64 (more machines than a warp has lanes, 64-bit machine masks), one edge group
    # per machine (E = M), a single job (the ESA mask's one-job branches), M = 2, J = 70 (three 32-job chunks), and
    # N = 143 (an odd size above one numpy pairwise leaf)
    ("j2m64e4_ls_esa_mixed", 2, 64, 4, 1, True, 1, "mixed", 1.0, 1, 111),
    ("j2m64e64_ls_fin_mixed", 2, 64, 64, 1, True, 0, "mixed", 1.0, 1, 112),
    ("j1m5e2_ls_esa_mixed", 1, 5, 2, 3, True, 1, "mixed", 1.0, 2, 113),
    ("j1m2e1_nols_fin_lowest", 1, 2, 1, 3, False, 0, "lowest", 1.0, 1, 114),
    ("j70m2e1_ls_esa_mixed", 70, 2, 1, 2, True, 1, "mixed", 1.0, 1, 115),
    ("j4m8e8_ls_esa_random", 4, 8, 8, 2, True, 1, "random", 1.0, 1, 116),
    ("j13m11e3_nols_esa_mixed", 13, 11, 3, 2, False, 1, "mixed", 1.0, 1, 117),
]
# steps whose full observation / schedule state a large fixture keeps (all steps below N = 200)
SPARSE_STEPS = sorted(set(range(0, 24)) | set(range(24, 600, 24)) | set(range(585, 600)))


def gen_replays(only=None):
    for (name, J, M, E, B, ls, mm, pol, scale, eps, seed) in REPLAYS:
        if only and name not in only:
            continue
        rng = np.random.default_rng(seed)
        if (J, M, E) == (6, 6, 2):
            d = ins.reference_stream_instances(100, 6, 6, 2, seed=1)  # shipped eval set
            idx = rng.choice(100, B, replace=False)
            d = {k: v[idx] for k, v in d.items()}
        else:
            d = ins.synthetic_instances(0, B, J, M, E, seed)
        t, p, tt, edge = d["t"] * scale, d["p"], d["transT"] * scale, d["edge"]
        w = rng.random((eps, B, 3))
        w = w / w.sum(-1, keepdims=True)
        r = rh.replay(J, M, E, t, p, tt, [edge[b] for b in range(B)], w, rng=rng, left_shift=ls, mask_mode=mm,
                      episodes=eps, machine_policy=pol, obs_steps=SPARSE_STEPS if J * M > 200 else None)
        adj = r.pop("adj"); adj0 = r.pop("adj0")
        assert np.array_equal(adj, adj.astype(np.int32)) and np.array_equal(adj0, adj0.astype(np.int32))
        out = dict(t=t, p=p, transT=tt, edge=edge, weights=w, J=J, M=M, E=E, left_shift=ls, mask_mode=mm,
                   adj=adj.astype(np.int32), adj0=adj0.astype(np.int32))
        out.update(r)
        out["actions"] = out["actions"].astype(np.int16); out["cand"] = out["cand"].astype(np.int16)
        out["mach"] = out["mach"].astype(np.int8); out["routes"] = out["routes"].astype(np.int16)
        path = os.path.join(HERE, "replay_%s.npz" % name)
        np.savez_compressed(path, **out)
        print(name, "%.0f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    import sys

    if len(sys.argv) > 1:  # python gen_golden.py replay_name ...: only those fixtures
        gen_replays(set(sys.argv[1:]))
    else:
        gen_pdr()
        gen_replays()
