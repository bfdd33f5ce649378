"""Samples of the reference's shipped instance pickles for tests/test_instances.py.

Run where a checkout of the reference project is available:

    MTFJSP_REFERENCE_ROOT=<reference checkout> python tests/golden/gen_instance_samples.py

Writes shipped_<stem>_first8.pkl: the first 8 instances of instance/<stem>.pkl in the same wire format (a pickled list
of the four arrays t, p, transT, edge, dtypes kept).  The whole files are pinned by the hashes in tests/test_instances.py,
checked here before writing.
"""
import hashlib
import os
import pickle
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_harness as rh  # noqa: E402
from tests.test_instances import SHIPPED  # noqa: E402

KEEP = 8


def main():
    for stem, (_, want) in SHIPPED.items():
        with open(os.path.join(rh.REF_ROOT, "instance", stem + ".pkl"), "rb") as f:
            arrays = pickle.load(f)
        got = tuple(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16] for a in arrays)
        assert got == want, (stem, got)
        with open(os.path.join(HERE, "shipped_%s_first%d.pkl" % (stem, KEEP)), "wb") as f:
            pickle.dump([np.ascontiguousarray(a[:KEEP]) for a in arrays], f)


if __name__ == "__main__":
    main()
