"""Golden data for sampled validation (PPO-S, the sampled-policy row of the reference's test table).

  csv16 [100,4]   row 16 (`PPO-S`) of results/test_results/Real_{MK,PT,TT,IT}_J6_M6_E2_Seed3_Weight442.csv: final
                  (makespan, processing energy / N, transport time, idle time) of the shipped `iotj` checkpoint rolled out
                  with greedy=False (test_all.py; one Categorical draw per actor per step, batch 1)
  csv13 [100,4]   row 13 (`MIP`) of the same files, the lower reference point of the quality table
Rows are 0-based as in gen_policy_golden.py.  The instances come from pdr_golden.npz and the `iotj` weights from
policy_golden.npz.  Run against a reference checkout: MTFJSP_REFERENCE_ROOT=<checkout> python gen_sampled_golden.py
"""
import csv
import os

import numpy as np

REF = os.environ.get("MTFJSP_REFERENCE_ROOT", "/root/reference")


def main():
    out = {}
    for row in (16, 13):
        a = np.zeros((100, 4))
        for k, name in enumerate(("MK", "PT", "TT", "IT")):
            rows = list(csv.reader(open(os.path.join(REF, "results/test_results/Real_%s_J6_M6_E2_Seed3_Weight442.csv" % name))))
            a[:, k] = [float(x) for x in rows[row][:100]]
        out["csv%d" % row] = a
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sampled_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()
