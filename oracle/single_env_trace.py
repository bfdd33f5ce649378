"""Recorded call sequences of the reference's single-env class, replayed on ours by tests/test_single_env.py.

TEST INFRASTRUCTURE ONLY.  tests/golden/gen_single_env_golden.py drives the reference class
(graph-jsp-env/.../disjunctive_graph_jsp_env_singlestep.py) the way the tests drive ours and stores, for every call,
the actions and a 64-bit digest of what the class returned (tests/golden/single_env_golden.npz).  A digest is taken of
a canonical form that two values share exactly when the tests' comparison calls them equal: arrays, lists and tuples
as float64 (with -0.0 folded into 0.0), numbers as float64, bools, strings and None by kind and value, dicts key by key,
DataFrames by columns, dtypes and values.
"""
from __future__ import annotations

import contextlib
import hashlib
import io

import numpy as np

STEP_CFGS = [(6, 6, 2, True, 3), (6, 6, 2, False, 4), (3, 4, 2, True, 5), (10, 10, 3, True, 6)]  # J, M, E, left shift, seed
PDR_ROWS = {(0, 0): 0, (0, 1): 1, (2, 0): 2, (5, 1): 9}   # (o_rule, m_rule) -> row of pdr_golden (CSV rows 0, 1, 4, 11)
PDR_INSTANCES = 12
VALIDATE_INSTANCES = 10


def cfg_key(cfg):
    J, M, E, ls, seed = cfg
    return "J%dM%dE%d_ls%d_s%d" % (J, M, E, int(ls), seed)


def _float_bytes(a):
    a = np.asarray(a, dtype=np.float64) + 0.0
    return repr(a.shape).encode() + np.where(np.isnan(a), np.nan, a).tobytes()


def canon(x, with_dtype=False) -> bytes:
    if isinstance(x, dict):
        return b"d{" + b",".join(repr(k).encode() + b":" + canon(x[k]) for k in sorted(x, key=repr)) + b"}"
    if type(x).__name__ == "DataFrame":
        df = x.reset_index(drop=True)
        parts = [b"df", repr(([str(c) for c in df.columns], [str(t) for t in df.dtypes])).encode()]
        for c in df.columns:
            col = df[c].to_numpy()
            parts.append(_float_bytes(col) if col.dtype.kind in "biuf" else repr([str(v) for v in col]).encode())
        return b"|".join(parts)
    if isinstance(x, (np.ndarray, list, tuple)):
        dt = np.asarray(x).dtype.str.encode() if with_dtype and isinstance(x, np.ndarray) else b""
        return b"a" + dt + _float_bytes(x)
    if isinstance(x, (bool, np.bool_)):
        return b"b1" if x else b"b0"
    if isinstance(x, str):
        return b"s" + x.encode()
    if x is None:
        return b"n"
    return b"f" + _float_bytes(float(x))


def digest(x, with_dtype=False) -> np.uint64:
    return np.frombuffer(hashlib.blake2b(canon(x, with_dtype), digest_size=8).digest(), dtype=np.uint64)[0]


def tuple_digests(tup):
    """One digest per element; the first element (the flat state vector) also carries its dtype."""
    return np.array([digest(v, with_dtype=(k == 0)) for k, v in enumerate(tup)], dtype=np.uint64)


def combined_digest(tup):
    return np.frombuffer(hashlib.blake2b(tuple_digests(tup).tobytes(), digest_size=8).digest(), dtype=np.uint64)[0]


def nodes_digest(env, N):
    """Node attributes the callers read: machine, scheduled, finish_time, job, duration, and start_time once scheduled."""
    rows = []
    for task_id in range(1, N + 1):
        n = env.G.nodes[task_id]
        rows.append([n[k] for k in ("machine", "scheduled", "finish_time", "job", "duration")] +
                    [n["start_time"] if n["scheduled"] else None])
    none = np.array([[v is None for v in r] for r in rows])
    vals = np.array([[np.nan if v is None else float(v) for v in r] for r in rows])
    return digest(np.concatenate([none.astype(np.float64), np.nan_to_num(vals, nan=0.0)]))


def routes_digest(env, M):
    r = [np.asarray(env.machine_routes[m], dtype=np.int64) for m in range(M)]
    return digest(np.concatenate([[len(x)] for x in r] + r).astype(np.float64))


def make_env(cls, t, p, tt, args, left_shift):
    with contextlib.redirect_stdout(io.StringIO()):
        return cls(jps_instance=np.array([t, p]), reward_function_parameters=args["reward_scaling"],
                   default_visualisations=["gantt_console", "graph_console"], reward_function="wrk", ability_tr_mm=tt,
                   perform_left_shift_if_possible=left_shift, configs=args)


def step_quiet(env, action):
    with contextlib.redirect_stdout(io.StringIO()):
        return env.step(joint_action=[int(action[0]), int(action[1])])


def final_costs(env, n_total_task):
    """What the rule rollout and the validation loop read once an episode is done: [mk, mean e1, transT, idleT]."""
    return [env.makespan_previous_step, env.total_e1_previous_step / n_total_task, env.trans_t_previous_step,
            env.idle_t_previous_step]
