"""Steepest-descent local search over finished schedules, on the environment's whole-episode replay
(BatchedMTFJSPEnv.replay, mtfjsp_replay).

This is the project's own improvement method; the reference has none (its test table compares constructive results with
the MIP solutions).  A schedule is the complete, valid action sequence a = [(o_s, m_s)], s = 0 .. N-1, that a constructive
method returns (greedy_validate, beam_validate, the rules' rollouts).  Its neighbourhood is every sequence one move away:

  reassignment (s, m')  step s runs on machine m' instead: m' is feasible for o_s (t >= 0) and m' != m_s;
  insertion    (s, s')  entry s is removed and inserted at index s' of the remaining N-1 entries, strictly after o_s's job
                        predecessor and strictly before its job successor (so every neighbour is a valid sequence), with
                        s' not in {s, s-1}: s is the identity, and s-1 gives the adjacent swap that (s-1, s) already gives.

The moves of an instance are ordered reassignments in (s, m') order, then insertions in (s, s') order; that order breaks
ties.  One round replays every neighbour of every instance from its episode start and, per instance, moves to the
neighbour of the lowest FP64 objective w_mk*mk + w_ec*(pt + idle) + w_tt*tt if that is strictly lower than the
incumbent's.  The search stops after `rounds` rounds or at the first round in which no instance moves: one host
synchronisation per round.  The environment decides what a sequence costs, so a neighbour's objective is exactly what
stepping it would give, left shift included.

`tabu_search` walks the same neighbourhood past local optima: every iteration it moves to the best neighbour that is not
tabu, improving or not, and a short memory of recent moves keeps it from walking straight back.  Neighbours are
replayed from the incumbent and the move list (BatchedMTFJSPEnv.replay_moves, mtfjsp_replay_moves) without being built,
and the move decision is one launch for every instance (mtfjsp_tabu_move).

`anneal_search` is parallel tempering on the same neighbourhood: K Markov chains per instance, each at its own
temperature, propose one uniformly drawn neighbour each per iteration (mtfjsp_anneal_propose), replay only that, take it
by the Metropolis rule and exchange states between adjacent temperatures (mtfjsp_anneal_step).  It spends one replay per
proposal where tabu search spends a whole neighbourhood per move.

`pareto_local_search` walks the same neighbourhood without a weighted sum: it keeps an archive of mutually
non-dominated schedules per instance over the three targets (pareto.py) and expands it until no member is left
unexplored.

`pilot_search` is constructive instead: the rollout algorithm (pilot method) on the environment's episode completion
(BatchedMTFJSPEnv.complete, mtfjsp_complete).  At every decision it lets a base heuristic finish the schedule after each
candidate action and takes the candidate whose completion is best.
"""
from __future__ import annotations

import numpy as np
import torch

from . import pareto
from ._lib import _ptr, _stream, check, lib
from .env import MASK_ESA, MASK_FINISHED, BatchedMTFJSPEnv
from .rules import priority_table
from .validate import _objective

REASSIGN, INSERT = 0, 1


def neighbour_moves(actions, t, max_neighbours=None, seed=0, round_=0):
    """All single moves of every instance's sequence, as a flat [R,4] int64 list of (instance, kind, s, arg) on the
    device of `actions`: kind REASSIGN with arg = the new machine m', kind INSERT with arg = the insertion index s'.
    Moves are grouped by instance in instance order, then in the tie order of the module docstring.
    actions: [N,S,2] integer (op, machine) sequences; t: [S,N,M] processing times (t < 0: infeasible), any device.
    max_neighbours: an instance with more moves keeps a uniform sample of that many, without replacement, in move
    order; the sample is a function of (seed, round_, max_neighbours) and of the move counts of the batch."""
    dev = actions.device
    a = actions.to(device=dev, dtype=torch.int64)
    t = torch.as_tensor(t).to(dev)
    N, S = a.shape[0], a.shape[1]
    M = t.shape[2]
    op, mach = a[..., 0].t(), a[..., 1].t()                                    # [S,N]
    inst = torch.arange(S, device=dev)
    # reassignments: (i, s, m') with t[i, o_s, m'] >= 0 and m' != m_s
    feas = (t[inst[:, None], op] >= 0) & (torch.arange(M, device=dev) != mach[..., None])   # [S,N,M]
    ri, rs, rm = feas.nonzero(as_tuple=True)
    # insertions: s' in (pos of the job predecessor, pos of the job successor), s' not in {s, s-1}
    pos = torch.empty_like(op)
    pos.scatter_(1, op, torch.arange(N, device=dev).expand(S, N))              # pos[i, o] = index of op o
    k = op % M
    pred = torch.where(k > 0, torch.gather(pos, 1, torch.clamp(op - 1, min=0)), -1)
    succ = torch.where(k < M - 1, torch.gather(pos, 1, torch.clamp(op + 1, max=N - 1)), N)
    sp = torch.arange(N, device=dev)                                           # s' over the N insertion indices
    s_ = torch.arange(N, device=dev)[:, None]
    ok = (sp > pred[..., None]) & (sp < succ[..., None]) & (sp != s_) & (sp != s_ - 1)      # [S,N,N]
    ii, is_, isp = ok.nonzero(as_tuple=True)
    moves = torch.cat((torch.stack((ri, torch.full_like(ri, REASSIGN), rs, rm), 1),
                       torch.stack((ii, torch.full_like(ii, INSERT), is_, isp), 1)))
    moves = moves[torch.sort(moves[:, 0] * 2 + moves[:, 1], stable=True)[1]]
    if max_neighbours is not None and moves.shape[0]:
        K = int(max_neighbours)
        if K < 1:
            raise ValueError("max_neighbours must be >= 1")
        state = np.random.SeedSequence([int(seed), int(round_), K]).generate_state(1, dtype=np.uint64)[0]
        g = torch.Generator().manual_seed(int(state) & 0x7FFFFFFFFFFFFFFF)
        key = torch.rand(moves.shape[0], generator=g, dtype=torch.float64).to(dev)
        # rank of every move among its instance's moves by random key: sort by key, then stably by instance
        o1 = torch.sort(key)[1]
        order = o1[torch.sort(moves[o1, 0], stable=True)[1]]
        count = torch.bincount(moves[:, 0], minlength=S)
        start = torch.cumsum(count, 0) - count
        rank = torch.empty_like(order)
        rank[order] = torch.arange(order.shape[0], device=dev) - start[moves[order, 0]]
        moves = moves[rank < K]
    return moves


def apply_moves(actions, moves):
    """The neighbour sequences of `moves` ([R,4] from neighbour_moves): [N,R,2] int32 on the device of `actions`, row r
    = actions[:, moves[r, 0]] with move r applied.  Index arithmetic only."""
    N = actions.shape[0]
    mv = moves.to(actions.device)
    i, kind, s, arg = mv[:, 0], mv[:, 1], mv[:, 2], mv[:, 3]
    base = actions.index_select(1, i)                                          # [N,R,2]
    n = torch.arange(N, device=actions.device)[:, None]
    ins = kind == INSERT
    sp = torch.where(ins, arg, 0)
    rest = torch.where(n < sp, n, n - 1)                                       # index in the remaining N-1 entries
    src = torch.where(rest < s, rest, rest + 1)
    src = torch.where(n == sp, s, src)
    src = torch.where(ins, src, n)                                             # [N,R]
    out = torch.gather(base, 0, src[..., None].expand(N, -1, 2)).to(torch.int32)
    re = (~ins).nonzero(as_tuple=True)[0]
    out[s[re], re, 1] = arg[re].to(torch.int32)
    return out


def local_search(instances, actions, weights=(0.4, 0.4, 0.2), left_shift=True, rounds=200, max_neighbours=None, seed=0,
                 max_candidates=65536, device=None):
    """Steepest descent from the S sequences `actions` ([N,S,2] integers, numpy or torch: complete valid schedules of
    the instances {"t","p","transT","edge"} [S,...]) under the reward weights `weights`.
    Neighbours are replayed on one env handle of the S instances (src = their instance), at most `max_candidates` per
    replay call.  With max_neighbours=None the result of an instance depends neither on max_candidates nor on the other
    instances of the batch.
    -> dict of numpy arrays: actions [N,S,2] int32, final4 [S,4], objective [S], history [rounds_run+1, S] (objective
    after each round, the start first; never increasing), accepted [rounds_run, S] bool, and replays, the number of
    sequences replayed (the start included)."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    if max_candidates < 1:
        raise ValueError("max_candidates must be >= 1")
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32)
    dev = env.device
    env.load(*(np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    cur = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).to(dev, torch.int32)
    if tuple(cur.shape) != (N, S, 2):
        raise ValueError("actions must have shape [%d, %d, 2]" % (N, S))
    t_dev = torch.as_tensor(t, device=dev)
    final4, _, finv = env.replay(cur)
    if bool((finv != -1).any()):
        raise ValueError("a starting sequence has an invalid action")
    obj = _objective(final4, weights)
    history, accepted = [obj], []
    replays = S
    inst_ids = torch.arange(S, device=dev)
    for rnd in range(int(rounds)):
        moves = neighbour_moves(cur, t_dev, max_neighbours, seed, rnd)
        R = moves.shape[0]
        replays += R
        f4 = torch.empty((R, 4), dtype=torch.float64, device=dev)
        bad = torch.zeros((), dtype=torch.bool, device=dev)
        for c0 in range(0, R, max_candidates):
            mv = moves[c0:c0 + max_candidates]
            f4[c0:c0 + mv.shape[0]], _, fi = env.replay(apply_moves(cur, mv), mv[:, 0].to(torch.int32))
            bad |= (fi != -1).any()
        o = _objective(f4, weights)
        mi = moves[:, 0]
        best = torch.full((S,), float("inf"), dtype=torch.float64, device=dev).scatter_reduce(0, mi, o, "amin")
        idx = torch.where(o == best[mi], torch.arange(R, device=dev), R)
        first = torch.full((S,), R, dtype=torch.int64, device=dev).scatter_reduce(0, mi, idx, "amin")
        acc = best < obj
        pick = torch.clamp(first, max=max(R - 1, 0))
        if R:
            chosen = moves[pick]
            chosen[:, 0] = inst_ids  # non-accepting instances: any move of their own, discarded below
            cur = torch.where(acc[None, :, None], apply_moves(cur, chosen), cur)
            final4 = torch.where(acc[:, None], f4[pick], final4)
        obj = torch.where(acc, best, obj)
        history.append(obj)
        accepted.append(acc)
        flags = torch.stack((acc.any(), bad)).cpu()
        if bool(flags[1]):
            raise RuntimeError("a neighbour replayed with an invalid action")
        if not bool(flags[0]):
            break
    env.close()
    return {"actions": cur.cpu().numpy(), "final4": final4.cpu().numpy(), "objective": obj.cpu().numpy(),
            "history": torch.stack(history).cpu().numpy(),
            "accepted": (torch.stack(accepted) if accepted else torch.zeros((0, S), dtype=torch.bool)).cpu().numpy(),
            "replays": replays}


# ---- tabu search on the neighbour replay -------------------------------------------------------------------------------
# the defaults come from a sweep on device-generated J6M6E2 instances (profiles/README.md, "Tabu search" (d))
TENURE_MACH, TENURE_INS = 20, 80
_TABU_STATE = ("cur", "cur_obj", "cur_f4", "best", "best_obj", "best_f4", "mach_until", "op_until")


def tabu_state(cur, f4, weights, M):
    """A fresh tabu state of S instances at the sequences cur ([S,N,2] int32) of final costs f4 ([S,4] f64), in the form
    mtfjsp_tabu_move updates: cur, cur_obj, cur_f4, best (= cur), best_obj, best_f4, mach_until [S,N,M] and op_until
    [S,N] int32 (all 0: nothing tabu).  Torch tensors on cur's device, or numpy arrays for numpy input."""
    if isinstance(cur, np.ndarray):
        xp, kw, cp = np, {}, np.copy
    else:
        xp, kw, cp = torch, {"device": cur.device}, torch.clone
    S, N = cur.shape[0], cur.shape[1]
    obj = _objective(f4, weights)
    return {"cur": cp(cur), "cur_obj": cp(obj), "cur_f4": cp(f4), "best": cp(cur), "best_obj": cp(obj), "best_f4": cp(f4),
            "mach_until": xp.zeros((S, N, M), dtype=xp.int32, **kw), "op_until": xp.zeros((S, N), dtype=xp.int32, **kw)}


def tabu_move(state, moves, seg, obj, f4, it, tenure_mach=TENURE_MACH, tenure_ins=TENURE_INS):
    """One tabu iteration's move for every instance on the device (mtfjsp_tabu_move; rules in include/mtfjsp.h): state
    as tabu_state returns it, updated in place; moves [R,4] integers grouped by instance in neighbour_moves' order, seg
    [S+1] integers (instance s's moves are moves[seg[s]:seg[s+1]]), obj [R] and f4 [R,4] f64 their objectives and costs.
    -> chosen [S] int32: the move taken, -1 for none admissible, -2 for a malformed segment."""
    cur, mu = state["cur"], state["mach_until"]
    S, N, M = cur.shape[0], cur.shape[1], mu.shape[2]
    R = int(moves.shape[0])
    mv = moves.to(torch.int32).contiguous()
    sg = seg.to(torch.int64).contiguous()
    o = obj.to(torch.float64).contiguous()
    f = f4.to(torch.float64).contiguous()
    chosen = torch.empty((S,), dtype=torch.int32, device=cur.device)
    check(lib().mtfjsp_tabu_move(S, N // M, M, _ptr(mv if R else None), R, _ptr(sg), _ptr(o if R else None),
                                 _ptr(f if R else None), int(it), int(tenure_mach), int(tenure_ins),
                                 *(_ptr(state[k]) for k in _TABU_STATE), _ptr(chosen), _stream()), "mtfjsp_tabu_move")
    return chosen


def tabu_reference(state, moves, seg, obj, f4, it, tenure_mach=TENURE_MACH, tenure_ins=TENURE_INS):
    """numpy restatement of mtfjsp_tabu_move, move for move: state as tabu_state(..., numpy) (copied, not changed),
    moves [R,4], seg [S+1], obj [R], f4 [R,4].  -> (the state after the move, chosen [S] int32)."""
    st = {k: np.array(v, copy=True) for k, v in state.items()}
    moves, seg = np.asarray(moves, dtype=np.int64), np.asarray(seg, dtype=np.int64)
    obj, f4 = np.asarray(obj, dtype=np.float64), np.asarray(f4, dtype=np.float64)
    S, N, M = st["cur"].shape[0], st["cur"].shape[1], st["mach_until"].shape[2]
    R = moves.shape[0]
    chosen = np.empty(S, dtype=np.int32)
    for s in range(S):
        lo, hi = int(seg[s]), int(seg[s + 1])
        if lo < 0 or hi < lo or hi > R:
            chosen[s] = -2
            continue
        row = st["cur"][s].copy()
        bo = st["best_obj"][s]
        bi, v = -1, None
        for r in range(lo, hi):
            i, kind, ms, arg = (int(x) for x in moves[r])
            if i != s or not 0 <= ms < N or not 0 <= row[ms, 0] < N:
                continue
            o = int(row[ms, 0])
            if kind == REASSIGN:
                if not (0 <= arg < M and 0 <= row[ms, 1] < M):
                    continue
                tabu = st["mach_until"][s, o, arg] > it
            elif kind == INSERT:
                if not 0 <= arg < N:
                    continue
                tabu = st["op_until"][s, o] > it
            else:
                continue
            x = obj[r]
            if np.isnan(x) or (tabu and not x < bo):
                continue
            if bi < 0 or x < v:
                bi, v = r, x
        if bi < 0:
            chosen[s] = -1
            continue
        _, kind, ms, arg = (int(x) for x in moves[bi])
        o = int(row[ms, 0])
        if kind == INSERT:
            rest = np.delete(row, ms, axis=0)
            st["cur"][s] = np.insert(rest, arg, row[ms], axis=0)
            st["op_until"][s, o] = it + 1 + tenure_ins
        else:
            st["cur"][s, ms, 1] = arg
            st["mach_until"][s, o, row[ms, 1]] = it + 1 + tenure_mach
        st["cur_obj"][s] = v
        st["cur_f4"][s] = f4[bi]
        if v < bo:
            st["best"][s] = st["cur"][s]
            st["best_obj"][s] = v
            st["best_f4"][s] = f4[bi]
        chosen[s] = bi
    return st, chosen


def tabu_search(instances, actions, weights=(0.4, 0.4, 0.2), left_shift=True, iterations=500, tenure_mach=TENURE_MACH,
                tenure_ins=TENURE_INS, max_neighbours=None, seed=0, max_candidates=65536, device=None):
    """Tabu search from the S sequences `actions` ([N,S,2] integers, numpy or torch: complete valid schedules of the
    instances {"t","p","transT","edge"} [S,...]) under the reward weights `weights`, on local_search's neighbourhood and
    FP64 objective.  Every iteration `it` runs neighbour_moves of the current sequences (max_neighbours samples as
    there, keyed by (seed, it)), replays them from the incumbent and the move list with BatchedMTFJSPEnv.replay_moves
    (src = their instance, at most max_candidates per call), and makes one mtfjsp_tabu_move: each instance moves to its
    admissible neighbour of the least objective, improving or not.  A reassignment of op o away from machine m makes
    (o, m) tabu for tenure_mach iterations; an insertion of o makes o's insertions tabu for tenure_ins iterations; a tabu
    move is admissible when it beats the instance's best (aspiration).  An instance with no admissible move stays put.
    Exactly `iterations` iterations run.  The histories stay on the device and the invalid-replay flag is read once, at
    the end; neighbour_moves' nonzero still synchronises once per iteration.

    While an instance descends, its current and best objectives are equal, so the steepest improving neighbour is
    admissible and wins with local_search's tie-break: with max_neighbours=None history follows local_search's history
    for as long as local_search accepts moves, and the result is never worse than local_search's.  With
    max_neighbours=None an instance's result depends neither on max_candidates nor on the other instances of the batch.
    -> dict of numpy arrays: actions [N,S,2] int32, final4 [S,4] and objective [S] of the best schedule, history
       [iterations+1, S] (the current objective, the start first), best_history [iterations+1, S] (never increasing),
       chosen [iterations, S] (mtfjsp_tabu_move's output) and replays, the number of sequences replayed (the start
       included)."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    if max_candidates < 1:
        raise ValueError("max_candidates must be >= 1")
    if int(iterations) < 0 or int(tenure_mach) < 0 or int(tenure_ins) < 0:
        raise ValueError("iterations and the tenures must be >= 0")
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32)
    dev = env.device
    env.load(*(np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    start = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).to(dev, torch.int32)
    if tuple(start.shape) != (N, S, 2):
        raise ValueError("actions must have shape [%d, %d, 2]" % (N, S))
    t_dev = torch.as_tensor(t, device=dev)
    final4, _, finv = env.replay(start)
    if bool((finv != -1).any()):
        raise ValueError("a starting sequence has an invalid action")
    st = tabu_state(start.transpose(0, 1).contiguous(), final4, weights, M)
    history, best_history, chosen = [st["cur_obj"].clone()], [st["best_obj"].clone()], []
    replays = S
    bad = torch.zeros((), dtype=torch.bool, device=dev)
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    for it in range(int(iterations)):
        base = st["cur"].transpose(0, 1)                                      # [N,S,2] view of the current sequences
        moves = neighbour_moves(base, t_dev, max_neighbours, seed, it)
        R = moves.shape[0]
        replays += R
        f4 = torch.empty((R, 4), dtype=torch.float64, device=dev)
        for c0 in range(0, R, max_candidates):
            mv = moves[c0:c0 + max_candidates]
            f4[c0:c0 + mv.shape[0]], _, fi = env.replay_moves(base, mv)
            bad |= (fi != -1).any()
        seg = torch.cat((zero, torch.cumsum(torch.bincount(moves[:, 0], minlength=S), 0)))
        chosen.append(tabu_move(st, moves, seg, _objective(f4, weights), f4, it, tenure_mach, tenure_ins))
        history.append(st["cur_obj"].clone())
        best_history.append(st["best_obj"].clone())
    if bool(bad):
        raise RuntimeError("a neighbour replayed with an invalid action")
    env.close()
    return {"actions": st["best"].transpose(0, 1).cpu().numpy(), "final4": st["best_f4"].cpu().numpy(),
            "objective": st["best_obj"].cpu().numpy(), "history": torch.stack(history).cpu().numpy(),
            "best_history": torch.stack(best_history).cpu().numpy(),
            "chosen": (torch.stack(chosen) if chosen else torch.zeros((0, S), dtype=torch.int32)).cpu().numpy(),
            "replays": replays}


# ---- parallel tempering on the neighbour replay ------------------------------------------------------------------------
# the defaults come from a sweep on device-generated J6M6E2 instances (profiles/README.md, "Parallel tempering" (a))
ANNEAL_CHAINS, ANNEAL_T_MAX, ANNEAL_T_MIN, ANNEAL_SWAP_EVERY = 32, 0.03, 1e-3, 1
_ANNEAL_STATE = ("cur", "cur_obj", "cur_f4", "best", "best_obj", "best_f4", "accepted", "swapped")
# exp_neg's constants (include/mtfjsp.h): Cody-Waite ln 2, 1/i! for the degree-13 Horner polynomial, the zero point
_INV_LN2, _LN2_HI, _LN2_LO, _EXP_NEG_ZERO = 1.4426950408889634, 0.6931471803691238, 1.9082149292705877e-10, 746.0
_INV_FACT = (1.0, 1.0, 0.5, 0.16666666666666666, 0.041666666666666664, 0.008333333333333333, 0.001388888888888889,
             0.0001984126984126984, 2.48015873015873e-05, 2.7557319223985893e-06, 2.755731922398589e-07,
             2.505210838544172e-08, 2.08767569878681e-09, 1.6059043836821613e-10)


def exp_neg_reference(x):
    """mtfjsp_anneal.cu's exp_neg in numpy, bit for bit: e^-x for x > 0, 1 for x <= 0, NaN for NaN, 0 past 746.  Cody-Waite
    reduction x = n ln2 + r, the degree-13 Taylor polynomial of e^z at z = -r in Horner form, and ldexp(p, -n)."""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        xc = np.where((x > 0.0) & (x <= _EXP_NEG_ZERO), x, 1.0)
        n = np.rint(xc * _INV_LN2)
        z = -((xc - n * _LN2_HI) - n * _LN2_LO)
        p = np.full_like(z, _INV_FACT[13])
        for c in _INV_FACT[12::-1]:
            p = p * z + c
        out = np.ldexp(p, -n.astype(np.int64))
    out = np.where(x <= 0.0, 1.0, np.where(x > _EXP_NEG_ZERO, 0.0, out))
    out = np.where(np.isnan(x), x, out)
    return out[()] if out.ndim == 0 else out


def anneal_ladder(K=ANNEAL_CHAINS, t_max=ANNEAL_T_MAX, t_min=ANNEAL_T_MIN):
    """The default ladder of K relative temperatures, ascending and geometric from t_min to t_max; K = 1 gives [t_max]."""
    K = int(K)
    if K < 1 or not 0 < t_min <= t_max or not np.isfinite(t_max):
        raise ValueError("anneal_ladder needs K >= 1 and 0 < t_min <= t_max < inf")
    if K == 1:
        return np.array([float(t_max)])
    lad = float(t_min) * (float(t_max) / float(t_min)) ** (np.arange(K) / (K - 1))
    lad[0], lad[-1] = t_min, t_max
    return np.maximum.accumulate(lad)


def anneal_state(cur, f4, weights, K):
    """A fresh annealing state of S instances with K chains each, every chain at its instance's sequence of cur ([S,N,2]
    int32) of final costs f4 ([S,4] f64), in the form mtfjsp_anneal_step updates: cur [S*K,N,2], cur_obj [S*K], cur_f4
    [S*K,4], best (= cur [S,N,2]), best_obj [S], best_f4 [S,4], and the per-call flags accepted [S*K] and swapped [S*K]
    int32.  Torch tensors on cur's device, or numpy arrays for numpy input."""
    if isinstance(cur, np.ndarray):
        xp, kw, cp, rep = np, {}, np.copy, lambda a: np.repeat(a, K, axis=0)
    else:
        xp, kw, cp, rep = torch, {"device": cur.device}, torch.clone, lambda a: torch.repeat_interleave(a, K, 0)
    S = cur.shape[0]
    obj = _objective(f4, weights)
    return {"cur": rep(cur), "cur_obj": rep(obj), "cur_f4": rep(f4), "best": cp(cur), "best_obj": cp(obj),
            "best_f4": cp(f4), "accepted": xp.zeros(S * K, dtype=xp.int32, **kw),
            "swapped": xp.zeros(S * K, dtype=xp.int32, **kw)}


def anneal_propose(t, cur, seed, it):
    """One uniformly drawn neighbour per chain on the device (mtfjsp_anneal_propose; rules in include/mtfjsp.h): t [S,N,M]
    f64 processing times, cur [S*K,N,2] int32 chain rows (row q = s*K + k), on one device.  -> moves [S*K,4] int32
    (row, kind, s, arg) in neighbour_moves' form, (q, -1, 0, 0) for a row without moves."""
    S, N, M = t.shape
    Q = int(cur.shape[0])
    if Q % S or tuple(cur.shape[1:]) != (N, 2):
        raise ValueError("cur must have shape [S*K, %d, 2]" % N)
    tt = t.to(torch.float64).contiguous()
    c = cur.to(torch.int32).contiguous()
    moves = torch.empty((Q, 4), dtype=torch.int32, device=cur.device)
    check(lib().mtfjsp_anneal_propose(_ptr(tt), S, N // M, M, Q // S, _ptr(c), int(seed) & 0xFFFFFFFFFFFFFFFF, int(it),
                                      _ptr(moves), _stream()), "mtfjsp_anneal_propose")
    return moves


def anneal_step(state, moves, first_invalid, obj, f4, temp, seed, it, swap_parity, M):
    """One iteration's Metropolis decisions, exchanges and best update on the device (mtfjsp_anneal_step; rules in
    include/mtfjsp.h): state as anneal_state returns it, updated in place (accepted and swapped rewritten); moves [S*K,4],
    first_invalid [S*K], obj [S*K] and f4 [S*K,4] the proposals' replay, temp [S,K] absolute temperatures; swap_parity 0
    or 1 exchanges the pairs (k, k+1) with k of that parity, anything else none; M the machine count (N = J*M)."""
    S, K = temp.shape
    N = state["cur"].shape[1]
    args = [x.to(dt).contiguous() for x, dt in ((moves, torch.int32), (first_invalid, torch.int32),
                                                 (obj, torch.float64), (f4, torch.float64), (temp, torch.float64))]
    check(lib().mtfjsp_anneal_step(S, N // M, M, K, *(_ptr(a) for a in args), int(seed) & 0xFFFFFFFFFFFFFFFF, int(it),
                                   int(swap_parity), *(_ptr(state[k]) for k in _ANNEAL_STATE), _stream()),
          "mtfjsp_anneal_step")


def anneal_propose_reference(t, cur, seed, it):
    """numpy restatement of mtfjsp_anneal_propose, draw for draw: row q's move is neighbour_moves(row q, t[s])
    [_below(u0, R_q)] with its row field set to q, (q, -1, 0, 0) when R_q = 0.  t [S,N,M], cur [S*K,N,2]; valid
    sequences only (the kernel's output for others is not restated)."""
    from .evolve import _below, _draws
    t = np.asarray(t, dtype=np.float64)
    cur = np.asarray(cur, dtype=np.int64)
    S, N, M = t.shape
    Q = cur.shape[0]
    K = Q // S
    inst = np.arange(Q) // K
    allm = neighbour_moves(torch.as_tensor(cur.transpose(1, 0, 2)), torch.as_tensor(t[inst])).numpy()
    count = np.bincount(allm[:, 0], minlength=Q)
    start = np.cumsum(count) - count
    out = np.zeros((Q, 4), dtype=np.int32)
    for q in range(Q):
        R = int(count[q])
        if R == 0:
            out[q] = (q, -1, 0, 0)
            continue
        u0 = _draws(seed, (int(it) << 32) | (q % K), 3)[0]
        out[q] = allm[start[q] + _below(u0, R)]
    return out


def anneal_step_reference(state, moves, first_invalid, obj, f4, temp, seed, it, swap_parity, M):
    """numpy restatement of mtfjsp_anneal_step, decision for decision: arguments as anneal_step, numpy; state copied, not
    changed.  -> the state after the step (accepted and swapped included)."""
    from .evolve import _draws
    st = {k: np.array(v, copy=True) for k, v in state.items()}
    moves, finv = np.asarray(moves, dtype=np.int64), np.asarray(first_invalid, dtype=np.int64)
    obj, f4, temp = (np.asarray(a, dtype=np.float64) for a in (obj, f4, temp))
    S, K = temp.shape
    N = st["cur"].shape[1]
    st["accepted"][:] = 0
    st["swapped"][:] = 0
    for s in range(S):
        u = [_draws(seed, (int(it) << 32) | k, 3) for k in range(K)]
        for k in range(K):
            q = s * K + k
            row, kind, ms, arg = (int(x) for x in moves[q])
            ok = row == q and kind in (REASSIGN, INSERT) and 0 <= ms < N and finv[q] == -1
            if ok:
                o, mo = (int(x) for x in st["cur"][q, ms])
                ok = 0 <= o < N and ((0 <= arg < M and 0 <= mo < M) if kind == REASSIGN else 0 <= arg < N)
            if not ok or np.isnan(obj[q]):
                continue
            delta, T = obj[q] - st["cur_obj"][q], temp[s, k]
            if not (delta <= 0.0 or (T > 0.0 and u[k][1] < exp_neg_reference(delta / T))):
                continue
            if kind == INSERT:
                r = st["cur"][q]
                st["cur"][q] = np.insert(np.delete(r, ms, axis=0), arg, r[ms], axis=0)
            else:
                st["cur"][q, ms, 1] = arg
            st["cur_obj"][q], st["cur_f4"][q] = obj[q], f4[q]
            st["accepted"][q] = 1
        if swap_parity in (0, 1):
            for k in range(int(swap_parity), K - 1, 2):
                a, b = s * K + k, s * K + k + 1
                d, Ta, Tb = st["cur_obj"][b] - st["cur_obj"][a], temp[s, k], temp[s, k + 1]
                with np.errstate(divide="ignore", invalid="ignore"):
                    swap = d <= 0.0 or (Ta > 0.0 and u[k][2] < exp_neg_reference(d * (1.0 / Ta - 1.0 / Tb)))
                if swap:
                    for key in ("cur", "cur_obj", "cur_f4"):
                        st[key][[a, b]] = st[key][[b, a]]
                    st["swapped"][a] = 1
        v, bk = st["best_obj"][s], -1
        for k in range(K):
            if st["cur_obj"][s * K + k] < v:
                v, bk = st["cur_obj"][s * K + k], k
        if bk >= 0:
            st["best"][s], st["best_obj"][s], st["best_f4"][s] = st["cur"][s * K + bk], v, st["cur_f4"][s * K + bk]
    return st


def _swap_parity(it, swap_every):
    return (it // swap_every) % 2 if swap_every > 0 and (it + 1) % swap_every == 0 else -1


def _check_ladder(ladder):
    lad = np.asarray(ladder, dtype=np.float64)
    if lad.ndim != 1 or lad.shape[0] < 1 or not np.isfinite(lad).all() or (lad < 0).any() or (np.diff(lad) < 0).any():
        raise ValueError("ladder must be a non-empty 1-D array of finite, nonnegative, nondecreasing temperatures")
    return lad


def anneal_search(instances, actions, weights=(0.4, 0.4, 0.2), left_shift=True, iterations=2000, ladder=None,
                  swap_every=ANNEAL_SWAP_EVERY, seed=0, max_candidates=65536, device=None):
    """Parallel tempering (replica-exchange simulated annealing) from the S sequences `actions` ([N,S,2] integers, numpy
    or torch: complete valid schedules of the instances {"t","p","transT","edge"} [S,...]) under the reward weights
    `weights`, on local_search's neighbourhood and FP64 objective.  Each instance runs K = len(ladder) chains, all starting
    from its sequence, chain k at the absolute temperature ladder[k] * the start objective (ladder: relative temperatures,
    finite, >= 0 and nondecreasing; None is anneal_ladder()'s defaults).  Every iteration `it` runs one anneal_propose (one
    uniform neighbour per chain), BatchedMTFJSPEnv.replay_moves of the S*K proposals (src = their instance, at most
    max_candidates per call), and one anneal_step: the Metropolis test per chain, then, on iterations with
    (it + 1) % swap_every == 0, exchanges of the adjacent pairs (k, k+1) with k = (it // swap_every) % 2 (mod 2);
    swap_every = 0 never exchanges.  Exactly `iterations` iterations run with no host synchronisation; the invalid-replay
    flag is read once, at the end.  Draws are keyed by (seed, it, k) only, so an instance's result depends neither on
    max_candidates nor on the other instances of the batch or its row in it.
    -> dict of numpy arrays: actions [N,S,2] int32, final4 [S,4] and objective [S] of the best schedule visited,
       best_history [iterations+1, S] (never increasing, the start first), current [S,K] (the chains' final objectives),
       accept_rate [K] (per rung, over instances and iterations), swap_rate [K-1] (per adjacent pair, over instances and
       the iterations that tried it; NaN if none did) and replays, the number of sequences replayed (the start
       included)."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    lad = anneal_ladder() if ladder is None else _check_ladder(ladder)
    K = lad.shape[0]
    if max_candidates < 1:
        raise ValueError("max_candidates must be >= 1")
    if int(iterations) < 0 or int(swap_every) < 0:
        raise ValueError("iterations and swap_every must be >= 0")
    if tuple(actions.shape if torch.is_tensor(actions) else np.shape(actions)) != (N, S, 2):
        raise ValueError("actions must have shape [%d, %d, 2]" % (N, S))
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32)
    dev = env.device
    start = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).to(dev, torch.int32)
    env.load(*(np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    t_dev = torch.as_tensor(t, device=dev, dtype=torch.float64)
    final4, _, finv = env.replay(start)
    if bool((finv != -1).any()):
        raise ValueError("a starting sequence has an invalid action")
    st = anneal_state(start.transpose(0, 1).contiguous(), final4, weights, K)
    temp = torch.as_tensor(lad, device=dev)[None, :] * st["best_obj"][:, None]                 # [S,K]
    Q = S * K
    row_src = torch.arange(Q, dtype=torch.int32, device=dev) // K                 # chain row -> its instance's env
    best_history = [st["best_obj"].clone()]
    acc_sum = torch.zeros(Q, dtype=torch.int64, device=dev)
    swap_sum = torch.zeros(Q, dtype=torch.int64, device=dev)
    tries = np.zeros(2, dtype=np.int64)                                            # exchanges tried per parity
    bad = torch.zeros((), dtype=torch.bool, device=dev)
    f4 = torch.empty((Q, 4), dtype=torch.float64, device=dev)
    fi = torch.empty((Q,), dtype=torch.int32, device=dev)
    for it in range(int(iterations)):
        moves = anneal_propose(t_dev, st["cur"], seed, it)
        base = st["cur"].transpose(0, 1)                                           # [N,S*K,2] view of the chain rows
        for c0 in range(0, Q, max_candidates):
            c1 = min(c0 + max_candidates, Q)
            f4[c0:c1], _, fi[c0:c1] = env.replay_moves(base, moves[c0:c1], row_src)
        bad |= (fi >= 0).any()
        par = _swap_parity(it, int(swap_every))
        if par >= 0:
            tries[par] += 1
        anneal_step(st, moves, fi, _objective(f4, weights), f4, temp, seed, it, par, M)
        acc_sum += st["accepted"]
        swap_sum += st["swapped"]
        best_history.append(st["best_obj"].clone())
    if bool(bad):
        raise RuntimeError("a neighbour replayed with an invalid action")
    env.close()
    pair_tries = tries[np.arange(K - 1) % 2] * S
    sw = swap_sum.view(S, K)[:, :K - 1].sum(0).cpu().numpy().astype(np.float64)
    acc = acc_sum.view(S, K).sum(0).cpu().numpy().astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        swap_rate = np.where(pair_tries > 0, sw / pair_tries, np.nan)
        accept_rate = acc / float(S * int(iterations))
    return {"actions": st["best"].transpose(0, 1).cpu().numpy(), "final4": st["best_f4"].cpu().numpy(),
            "objective": st["best_obj"].cpu().numpy(), "best_history": torch.stack(best_history).cpu().numpy(),
            "current": st["cur_obj"].view(S, K).cpu().numpy(),
            "accept_rate": accept_rate, "swap_rate": swap_rate, "replays": S + int(iterations) * Q}


def _replay_all(env, R, seqs, src, max_candidates):
    """final4 [R,4] of R sequences, each replayed from the episode start of env src[r] ([R] int32), at most
    max_candidates per replay call; seqs(c0, c1) builds the [N, c1 - c0, 2] sequences of candidates c0 .. c1 - 1.
    Also a device flag: some action was invalid."""
    f4 = torch.empty((R, 4), dtype=torch.float64, device=env.device)
    bad = torch.zeros((), dtype=torch.bool, device=env.device)
    for c0 in range(0, R, max_candidates):
        c1 = min(R, c0 + max_candidates)
        f4[c0:c1], _, fi = env.replay(seqs(c0, c1), src[c0:c1])
        bad |= (fi != -1).any()
    return f4, bad


def _merge(count, arch_f4, new_inst, new_f4, cap):
    """One archive-first merge.  The archive (arch_f4 [S,A,4], the first count[s] slots of row s valid) in archive order,
    then the new points (new_f4 [R,4] of instances new_inst [R], grouped by instance in candidate order), per instance;
    filtered by mtfjsp_pareto_filter, fronts of more than `cap` points cut by crowding distance.
    -> survivors in merged order as (is_new, index: archive flat index s * A + a or new candidate index, instance, slot),
       their count [S] and truncated [S] bool."""
    S, A = arch_f4.shape[0], arch_f4.shape[1]
    dev = arch_f4.device
    oi, oa = (torch.arange(A, device=dev)[None, :] < count[:, None]).nonzero(as_tuple=True)
    inst = torch.cat((oi, new_inst))
    is_new = torch.cat((torch.zeros_like(oi, dtype=torch.bool), torch.ones_like(new_inst, dtype=torch.bool)))
    idx = torch.cat((oi * A + oa, torch.arange(new_inst.shape[0], device=dev)))
    order = torch.sort(inst * 2 + is_new.long(), stable=True)[1]            # instance; the archive first; list order
    inst, is_new, idx = inst[order], is_new[order], idx[order]
    obj = pareto.objectives(torch.cat((arch_f4.view(S * A, 4)[oi * A + oa], new_f4))[order])
    cnt = torch.bincount(inst, minlength=S)
    seg = torch.cat((torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(cnt, 0)))
    keep = pareto.pareto_filter(obj, seg, max_len=inst.shape[0])
    inst, is_new, idx, obj = inst[keep], is_new[keep], idx[keep], obj[keep]
    truncated = torch.bincount(inst, minlength=S) > cap
    cut = pareto.crowding_truncate(obj, inst, S, cap)
    inst, is_new, idx = inst[cut], is_new[cut], idx[cut]
    count = torch.bincount(inst, minlength=S)
    slot = torch.arange(inst.shape[0], device=dev) - (torch.cumsum(count, 0) - count)[inst]
    return is_new, idx, inst, slot, count, truncated


def pareto_local_search(instances, actions, weights=(0.4, 0.4, 0.2), left_shift=True, rounds=200, expand=8,
                        max_archive=256, max_neighbours=None, seed=0, max_candidates=65536, device=None):
    """Pareto local search over the three targets (mk, ec = pt + idle, tt; pareto.objectives) from the start sequences
    `actions` ([N,S,2] or [N,K,S,2] integers, numpy or torch: complete valid schedules of the instances
    {"t","p","transT","edge"} [S,...]).

    Each instance keeps an archive of mutually non-dominated schedules, at most `max_archive` (<= 4,096) of them.  The
    start set is filtered into it in k order.  Each round, per instance, the first `expand` unexplored members in archive
    order are marked explored, and their neighbourhoods (neighbour_moves with each member as one column; max_neighbours
    samples as there) are replayed from the instance's episode start, at most `max_candidates` per replay call.  The
    archive in archive order, then the neighbours in (member, move) order, go through mtfjsp_pareto_filter, which keeps
    the first of equal cost vectors: an archive member beats a neighbour of the same costs.  New survivors start
    unexplored.  A front of more than max_archive points keeps the max_archive of the largest crowding distance
    (pareto.crowding_truncate); survivors keep their merged order.  The search stops when no instance has an unexplored
    member, or after `rounds` rounds: one host synchronisation per round.  `weights` are the env's reward weights; they
    do not change the costs.  With max_neighbours=None the result of an instance depends neither on max_candidates nor
    on the other instances of the batch.
    -> dict of numpy arrays, A = max_archive: actions [N,S,A,2] int32 (-1 past count), final4 [S,A,4] and objectives
       [S,A,3] (NaN past count), count [S], explored [S,A] bool, ref [S,3] (1.1 x the componentwise max of the start
       set's objectives, 1.0 where that max is 0), hypervolume [rounds_run+1, S] (the archive's in ref, the start first),
       truncated [rounds_run, S] bool, and replays, the number of candidates replayed (the start set included)."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    A = int(max_archive)
    if max_candidates < 1 or expand < 1 or not 1 <= A <= pareto.HV_MAX_POINTS:
        raise ValueError("max_candidates and expand must be >= 1, and 1 <= max_archive <= %d" % pareto.HV_MAX_POINTS)
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32)
    dev = env.device
    env.load(*(np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    start = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).to(dev, torch.int32)
    if start.dim() == 3:
        start = start[:, None]
    if start.dim() != 4 or (start.shape[0], start.shape[2], start.shape[3]) != (N, S, 2):
        raise ValueError("actions must have shape [%d, %d, 2] or [%d, K, %d, 2]" % (N, S, N, S))
    K = start.shape[1]
    start = start.transpose(1, 2).reshape(N, S * K, 2)                       # column s * K + k
    s_inst = torch.arange(S, device=dev).repeat_interleave(K)
    f4, bad = _replay_all(env, S * K, lambda a, b: start[:, a:b], s_inst.to(torch.int32), max_candidates)
    if bool(bad):
        raise ValueError("a starting sequence has an invalid action")
    replays = S * K
    ref = torch.as_tensor(pareto.reference_point(pareto.objectives(f4).view(S, K, 3).transpose(0, 1).cpu().numpy()),
                          device=dev)
    t_dev = torch.as_tensor(t, device=dev)
    arch_act = torch.full((N, S, A, 2), -1, dtype=torch.int32, device=dev)
    arch_f4 = torch.full((S, A, 4), float("nan"), dtype=torch.float64, device=dev)
    explored = torch.zeros((S, A), dtype=torch.bool, device=dev)
    count = torch.zeros((S,), dtype=torch.int64, device=dev)
    seg_a = torch.arange(S + 1, dtype=torch.int64, device=dev) * A

    def merge(new_inst, new_f4, new_seqs):
        nonlocal arch_act, arch_f4, explored, count
        is_new, idx, inst, slot, count, trunc = _merge(count, arch_f4, new_inst, new_f4, A)
        act2 = torch.full_like(arch_act, -1)
        f42 = torch.full_like(arch_f4, float("nan"))
        exp2 = torch.zeros_like(explored)
        o, n = ~is_new, is_new
        act2[:, inst[o], slot[o]] = arch_act.view(N, S * A, 2)[:, idx[o]]
        f42[inst[o], slot[o]] = arch_f4.view(S * A, 4)[idx[o]]
        exp2[inst[o], slot[o]] = explored.view(S * A)[idx[o]]
        act2[:, inst[n], slot[n]] = new_seqs(idx[n])
        f42[inst[n], slot[n]] = new_f4[idx[n]]
        arch_act, arch_f4, explored = act2, f42, exp2
        return trunc

    def archive_hv():
        return pareto.hypervolume(pareto.objectives(arch_f4).view(S * A, 3), seg_a, ref)

    merge(s_inst, f4, lambda i: start[:, i])
    history, truncated = [archive_hv()], []
    for rnd in range(int(rounds)):
        valid = torch.arange(A, device=dev)[None, :] < count[:, None]
        open_ = valid & ~explored
        pick = open_ & (torch.cumsum(open_.long(), 1) <= expand)             # the first `expand` unexplored members
        ms, ma = pick.nonzero(as_tuple=True)                                 # members in (instance, archive) order
        explored = explored | pick
        members = arch_act[:, ms, ma]                                        # [N,Msel,2], one member per column
        moves = neighbour_moves(members, t_dev[ms], max_neighbours, seed, rnd)
        nb_inst = ms[moves[:, 0]]
        f4n, badn = _replay_all(env, moves.shape[0], lambda a, b: apply_moves(members, moves[a:b]),
                                nb_inst.to(torch.int32), max_candidates)
        replays += int(moves.shape[0])
        truncated.append(merge(nb_inst, f4n, lambda i: apply_moves(members, moves[i])))
        history.append(archive_hv())
        valid = torch.arange(A, device=dev)[None, :] < count[:, None]
        flags = torch.stack(((valid & ~explored).any(), badn)).cpu()
        if bool(flags[1]):
            raise RuntimeError("a neighbour replayed with an invalid action")
        if not bool(flags[0]):
            break
    env.close()
    return {"actions": arch_act.cpu().numpy(), "final4": arch_f4.cpu().numpy(),
            "objectives": pareto.objectives(arch_f4).cpu().numpy(), "count": count.cpu().numpy(),
            "explored": explored.cpu().numpy(), "ref": ref.cpu().numpy(),
            "hypervolume": torch.stack(history).cpu().numpy(),
            "truncated": (torch.stack(truncated) if truncated else torch.zeros((0, S), dtype=torch.bool)).cpu().numpy(),
            "replays": replays}


def pilot_search(instances, base=("MWKR_T", "SPT"), candidates="all", weights=(0.4, 0.4, 0.2), left_shift=False,
                 mask_mode=MASK_FINISHED, samples=1, seed=0, max_candidates=65536, device=None):
    """The pilot method (rollout algorithm) on the instances {"t","p","transT","edge"} [S,...] under the reward weights
    `weights`, with a base heuristic finishing every candidate's schedule on the device (BatchedMTFJSPEnv.complete).

    base: an (operation rule, machine rule) pair of rules.OP_RULES x rules.MACHINE_RULES, run as its priority table
    (rules.priority_table), or "random" (policy_random's draws).  One live env of the S instances makes N decisions.  At
    each, the candidates of an instance are every (candidate op of a selectable job, machine) pair (candidates="all",
    flat index j*M + m) or the candidate op of every selectable job on the base rule's machine ("rule", flat index j;
    not for the random base); selectable means open under the `mask_mode` job mask.  One completion per candidate (T = 1,
    src = its instance; `samples` completions under the random base, the candidate scoring their minimum), at most
    `max_candidates` per call, scores it by the FP64 objective w_mk*mk + w_ec*(pt + idle) + w_tt*tt of its final costs;
    a candidate that is not selectable, or whose completion met an invalid action, scores +inf.  The lowest score wins,
    ties to the lowest flat index, and the live env steps it.  Each instance keeps an incumbent: the best complete
    sequence seen (ties keep the earlier), built from the pilot's prefix, the candidate and the base's actions.
    Shapes are static: no decision reads the device; there is one synchronisation at the end.

    With a deterministic base whose own choice is always a candidate (the priority base, under either candidate set),
    history never increases: the best completion's next action is a candidate at the next decision and completes to the
    same final state.  With the priority base an instance's result depends neither on the batch nor on max_candidates.
    With the random base the draws are keyed by (seed, decision, row of the completion call), so an instance's result
    depends on its row in the batch, as evolve.nsga2's does, and on max_candidates where that splits the candidates
    over several calls.  left_shift=False (the default) runs the rules as evaluate_rules does, so history[0] equals
    the rule's row there.
    -> dict: actions [N,S,2] int32 (the incumbents), final4 [S,4], objective [S] (= history.min(0)), history [N+1,S]
       (history[0] the base's own completion from the start, history[k+1] the best candidate score at decision k),
       base_objective [S] (= history[0]), completions (completion runs) and env_steps (steps they took)."""
    t = np.asarray(instances["t"], dtype=np.float64)
    p = np.asarray(instances["p"], dtype=np.float64)
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    Q = int(samples)
    if candidates not in ("all", "rule"):
        raise ValueError("candidates must be 'all' or 'rule'")
    if isinstance(base, str):
        if base != "random":
            raise ValueError("base must be 'random' or an (operation rule, machine rule) pair")
        if candidates == "rule":
            raise ValueError("candidates='rule' needs a rule pair as the base")
        kind = "random"
    else:
        kind = "priority"
        if Q != 1:
            raise ValueError("samples applies to the random base only")
    if Q < 1 or max_candidates < 1:
        raise ValueError("samples and max_candidates must be >= 1")
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32,
                           mask_mode=mask_mode)
    dev = env.device
    env.load(t, p, np.asarray(instances["transT"]), np.asarray(instances["edge"]))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    key = mach_tab = None
    if kind == "priority":
        k_np, m_np = priority_table(base[0], base[1], t, p, J, M)
        key, mach_tab = torch.as_tensor(k_np, device=dev), torch.as_tensor(m_np, device=dev)
    C = J * M if candidates == "all" else J
    inst = torch.arange(S, device=dev)
    env_steps = torch.zeros((), dtype=torch.int64, device=dev)
    completions = 0

    def best_completion(per, act, closed, k):
        """Completions of S * per rows, row r from instance r // per, forced actions act [T, S*per, 2] or None; closed
        [S*per] bool rows scoring +inf, or None.  -> per instance the lowest score, its row (the lowest of equal
        scores), final4 [S,4] and base actions [N,S,2]."""
        nonlocal env_steps, completions
        R = S * per
        ds = int(np.random.SeedSequence([int(seed), k]).generate_state(1, dtype=np.uint64)[0])
        src = torch.arange(R, device=dev, dtype=torch.int32) // per
        b_obj = torch.full((S,), float("inf"), dtype=torch.float64, device=dev)
        b_row = torch.zeros((S,), dtype=torch.int64, device=dev)
        b_f4 = torch.zeros((S, 4), dtype=torch.float64, device=dev)
        b_act = torch.full((N, S, 2), -1, dtype=torch.int32, device=dev)
        for c0 in range(0, R, max_candidates):
            c1 = min(R, c0 + max_candidates)
            f4, _, fi, ba = env.complete(src[c0:c1], None if act is None else act[:, c0:c1], base=kind, key=key,
                                         mach=mach_tab, seed=ds, mask_mode=mask_mode)
            T = 0 if act is None else act.shape[0]
            env_steps += (ba[..., 0] >= 0).sum() + T * (c1 - c0)
            ok = fi == -1
            if closed is not None:
                ok &= ~closed[c0:c1]
            o = torch.where(ok, _objective(f4, weights), float("inf"))
            si = src[c0:c1].long()
            cmin = torch.full((S,), float("inf"), dtype=torch.float64, device=dev).scatter_reduce(0, si, o, "amin")
            rows = torch.arange(c0, c1, device=dev)
            crow = torch.full((S,), R, dtype=torch.int64, device=dev).scatter_reduce(
                0, si, torch.where(o == cmin[si], rows, R), "amin")
            better = cmin < b_obj                                             # a later chunk's equal score has a later row
            loc = torch.clamp(crow - c0, 0, c1 - c0 - 1)
            b_obj = torch.where(better, cmin, b_obj)
            b_row = torch.where(better, crow, b_row)
            b_f4 = torch.where(better[:, None], f4[loc], b_f4)
            b_act = torch.where(better[None, :, None], ba[:, loc], b_act)
            completions += c1 - c0
        return b_obj, b_row, b_f4, b_act

    obj0, _, inc_f4, inc_act = best_completion(Q, None, None, 0)
    inc_obj = obj0
    history = [obj0]
    env.obs(mask_mode)
    acts = torch.full((N, S, 2), -1, dtype=torch.int32, device=dev)
    jj = torch.arange(C, device=dev) // M if candidates == "all" else torch.arange(C, device=dev)
    for k in range(N):
        cand = env.candidate                                                   # [S,J], current after obs / step_obs
        closed = env.job_mask.bool()
        op = cand[:, jj]                                                       # [S,C]
        if candidates == "all":
            mc = (torch.arange(C, device=dev) % M).to(torch.int32).expand(S, C)
        else:
            mc = torch.gather(mach_tab, 1, op.long())
        pair = torch.stack((op, mc), 2).repeat_interleave(Q, dim=1).reshape(1, S * C * Q, 2)
        cl = closed[:, jj].repeat_interleave(Q, dim=1).reshape(S * C * Q)
        b_obj, b_row, b_f4, b_act = best_completion(C * Q, pair, cl, k + 1)
        c = (b_row % (C * Q)) // Q
        a = torch.stack((op[inst, c], mc[inst, c]), 1)                         # [S,2]
        new = torch.cat((acts[:k], a[None], b_act[:N - k - 1]))
        better = b_obj < inc_obj
        inc_act = torch.where(better[None, :, None], new, inc_act)
        inc_f4 = torch.where(better[:, None], b_f4, inc_f4)
        inc_obj = torch.where(better, b_obj, inc_obj)
        history.append(b_obj)
        acts[k] = a
        env.step_obs(a[:, 0].contiguous(), a[:, 1].contiguous(), mask_mode)
    out = {"actions": inc_act.cpu().numpy(), "final4": inc_f4.cpu().numpy(), "objective": inc_obj.cpu().numpy(),
           "history": torch.stack(history).cpu().numpy(), "base_objective": obj0.cpu().numpy(),
           "completions": completions, "env_steps": int(env_steps.item())}
    env.close()
    return out


# ---- Monte Carlo tree search on the episode completion ------------------------------------------------------------------
# node fields of a tree pool (include/mtfjsp.h, mtfjsp_mcts_select)
PARENT, FIRST, NCHILD, OP, MACH, VISITS, VIRTUAL = range(7)


def mcts_trees(S, max_nodes, device=None):
    """S fresh trees of max_nodes nodes each, as mtfjsp_mcts_select / mtfjsp_mcts_backup read them: node [S,P,7] int32,
    vmin [S,P] f64, root [S] and count [S] int32, lohi [S,2] f64.  Node 0 is every tree's root; nothing is scored.
    device None: torch tensors on the current CUDA device; "numpy": numpy arrays (mcts_reference's form)."""
    P = int(max_nodes)
    if device == "numpy":
        xp, kw = np, {}
    else:
        xp, kw = torch, {"device": torch.device("cuda", torch.cuda.current_device()) if device is None else device}
    node = xp.zeros((S, P, 7), dtype=xp.int32, **kw)
    node[..., PARENT] = -1
    node[..., FIRST] = -1
    node[..., OP] = -1
    node[..., MACH] = -1
    lohi = xp.zeros((S, 2), dtype=xp.float64, **kw)
    lohi[:, 0], lohi[:, 1] = float("inf"), float("-inf")
    return {"node": node, "vmin": xp.full((S, P), float("inf"), dtype=xp.float64, **kw),
            "root": xp.zeros(S, dtype=xp.int32, **kw), "count": xp.ones(S, dtype=xp.int32, **kw), "lohi": lohi}


def mcts_select(t, next_op, tree, leaves, c, mach=None, max_depth=None):
    """One round of `leaves` selections per tree on the device (mtfjsp_mcts_select).  t [S,N,M] f64 and next_op [S,J]
    int32 (the root's next op index of every job, M when finished) on the trees' device; mach [S,N] int32 for the "rule"
    candidates, None for "all".  Updates `tree` in place.  -> paths [S*L, D, 2] int32 (D = max_depth, default N),
    depth [S*L] and leaf [S*L] int32."""
    node = tree["node"]
    S, P = node.shape[0], node.shape[1]
    N, M = t.shape[1], t.shape[2]
    J = N // M
    L, D = int(leaves), N if max_depth is None else int(max_depth)
    dev = node.device
    paths = torch.empty((S * L, D, 2), dtype=torch.int32, device=dev)
    depth = torch.empty((S * L,), dtype=torch.int32, device=dev)
    leaf = torch.empty((S * L,), dtype=torch.int32, device=dev)
    t = t.to(torch.float64).contiguous()
    nx = next_op.to(torch.int32).contiguous()
    m = None if mach is None else mach.to(torch.int32).contiguous()
    check(lib().mtfjsp_mcts_select(_ptr(t), _ptr(m), S, J, M, _ptr(nx), L, P, D, float(c), _ptr(node), _ptr(tree["vmin"]),
                                   _ptr(tree["root"]), _ptr(tree["count"]), _ptr(tree["lohi"]), _ptr(paths), _ptr(depth),
                                   _ptr(leaf), _stream()), "mtfjsp_mcts_select")
    return paths, depth, leaf


def mcts_backup(tree, leaf, objective):
    """Backs the round's S*L objectives (f64, +inf for a failed completion) up the paths ending at `leaf`
    (mtfjsp_mcts_backup).  Updates `tree` in place."""
    node = tree["node"]
    S, P = node.shape[0], node.shape[1]
    L = leaf.shape[0] // S
    obj = objective.to(torch.float64).contiguous()
    check(lib().mtfjsp_mcts_backup(S, L, P, _ptr(leaf), _ptr(obj), _ptr(node), _ptr(tree["vmin"]), _ptr(tree["root"]),
                                   _ptr(tree["count"]), _ptr(tree["lohi"]), _stream()), "mtfjsp_mcts_backup")


def _ref_children(ts, rule, nx, M):
    """(op, machine) children of a node, in flat-index order, from its per-job next op index nx."""
    out = []
    for j, k in enumerate(nx):
        if not 0 <= k < M:
            continue
        op = j * M + int(k)
        if rule is None:
            out += [(op, m) for m in range(M) if ts[op, m] >= 0.0]
        elif 0 <= rule[op] < M and ts[op, rule[op]] >= 0.0:
            out.append((op, int(rule[op])))
    return out


def _ref_select(t, next_op, tree, L, c, mach, D):
    node, vm, lohi = tree["node"], tree["vmin"], tree["lohi"]
    S, P = node.shape[0], node.shape[1]
    M = t.shape[2]
    N = t.shape[1]
    paths = np.full((S * L, D, 2), -1, dtype=np.int32)
    depth = np.zeros(S * L, dtype=np.int32)
    leaf = np.zeros(S * L, dtype=np.int32)
    for s in range(S):
        nd = node[s]
        lo, hi = lohi[s, 0], lohi[s, 1]
        cnt, r0 = int(tree["count"][s]), int(tree["root"][s])
        ok = 1 <= cnt <= P and 0 <= r0 < cnt
        for l in range(L):
            row = s * L + l
            nx = next_op[s].astype(np.int64).copy()
            x, d = (r0 if ok else -1), 0
            while x >= 0:
                seen = int(nd[x, VISITS]) + int(nd[x, VIRTUAL])
                fc, nc = int(nd[x, FIRST]), int(nd[x, NCHILD])
                nd[x, VIRTUAL] += 1
                if fc == -1 and nc == 0:
                    if seen == 0 or d >= D:
                        break
                    ch = _ref_children(t[s], None if mach is None else mach[s], nx, M)
                    if not ch or len(ch) > P - cnt:
                        break
                    for i, (op, m) in enumerate(ch):
                        nd[cnt + i] = (x, -1, 0, op, m, 0, 0)
                        vm[s, cnt + i] = np.inf
                    nd[x, FIRST], nd[x, NCHILD] = cnt, len(ch)
                    child = cnt
                    cnt += len(ch)
                else:
                    if fc < 0 or nc < 1 or fc > cnt - nc or d >= D:
                        break
                    n, v = nd[fc:fc + nc, VISITS].astype(np.int64), nd[fc:fc + nc, VIRTUAL].astype(np.int64)
                    fresh = np.nonzero(n + v == 0)[0]
                    if fresh.size:
                        child = fc + int(fresh[0])
                    else:
                        u = np.float64(c) * np.sqrt(np.float64(seen + 1))
                        best, bi = None, -1
                        for i in range(nc):
                            vc = vm[s, fc + i]
                            q = np.float64(0.0) if vc == np.inf else (np.float64(1.0) if hi == lo else (hi - vc) / (hi - lo))
                            sc = q * np.float64(n[i]) / np.float64(n[i] + v[i]) + u / np.float64(1 + n[i] + v[i])
                            if best is None or sc > best:
                                best, bi = sc, i
                        child = fc + bi
                op, m = int(nd[child, OP]), int(nd[child, MACH])
                paths[row, d] = (op, m)
                if 0 <= op < N:
                    nx[op // M] += 1
                d += 1
                x = child
            depth[row], leaf[row] = d, x
        tree["count"][s] = cnt
    return paths, depth, leaf


def _ref_backup(tree, leaf, obj):
    node, vm, lohi = tree["node"], tree["vmin"], tree["lohi"]
    S = node.shape[0]
    L = leaf.shape[0] // S
    for s in range(S):
        cnt, r0 = min(int(tree["count"][s]), node.shape[1]), int(tree["root"][s])
        for l in range(L):
            v, x = np.float64(obj[s * L + l]), int(leaf[s * L + l])
            if not 0 <= x < cnt:
                continue
            for _ in range(cnt):
                node[s, x, VISITS] += 1
                node[s, x, VIRTUAL] -= 1
                if v < vm[s, x]:
                    vm[s, x] = v
                if x == r0:
                    break
                x = int(node[s, x, PARENT])
                if not 0 <= x < cnt:
                    break
            if np.isfinite(v):
                lohi[s, 0] = min(lohi[s, 0], v)
                lohi[s, 1] = max(lohi[s, 1], v)


def mcts_reference(t, next_op, tree, leaves, c, objectives, mach=None, max_depth=None):
    """numpy restatement of mtfjsp_mcts_select and mtfjsp_mcts_backup (include/mtfjsp.h), bit for bit.  For every row of
    objectives ([R, S*L] f64) one round: `leaves` selections per tree, then the backup of that row.  t [S,N,M], next_op
    [S,J], mach [S,N] or None ("all"), tree as mcts_trees(..., device="numpy") returns it (copied, not changed).
    -> paths [R, S*L, D, 2], depth [R, S*L], leaf [R, S*L] (each round's selection) and the tree after the last backup."""
    t = np.asarray(t, dtype=np.float64)
    tree = {k: np.array(v, copy=True) for k, v in tree.items()}
    next_op = np.asarray(next_op)
    mach = None if mach is None else np.asarray(mach)
    D = t.shape[1] if max_depth is None else int(max_depth)
    out = []
    for obj in np.asarray(objectives, dtype=np.float64).reshape(-1, next_op.shape[0] * int(leaves)):
        out.append(_ref_select(t, next_op, tree, int(leaves), c, mach, D))
        _ref_backup(tree, out[-1][2], obj)
    paths, depth, leaf = (np.stack([o[i] for o in out]) for i in range(3))
    return paths, depth, leaf, tree


def mcts_search(instances, base=("MWKR_T", "SPT"), candidates="all", simulations=256, leaves=64, c=1.0,
                max_nodes=65536, weights=(0.4, 0.4, 0.2), left_shift=False, mask_mode=MASK_FINISHED, seed=0,
                max_candidates=65536, device=None):
    """Monte Carlo tree search over joint (op, machine) actions on the instances {"t","p","transT","edge"} [S,...] under
    the reward weights `weights`, with leaves scored by the device episode completion (BatchedMTFJSPEnv.complete).

    base and candidates are pilot_search's: an (operation rule, machine rule) pair run as its priority table, or
    "random"; children are every (candidate op of an open job, feasible machine) pair (candidates="all", flat index
    j*M + m) or the candidate op of every open job on the base rule's machine ("rule", flat index j; not for the random
    base).  Open means unfinished: only the FINISHED job mask is supported.  One tree per instance, a pool of max_nodes
    nodes (mcts_trees; 36 bytes a node).  One live env of the S instances makes N decisions.  Each decision runs
    ceil(simulations / leaves) rounds of `leaves` selections per tree (mtfjsp_mcts_select: unvisited children first in
    flat-index order, then the largest q*n/(n+v) + c*sqrt(Np+Vp)/(1+n+v) with q the child's best objective rescaled to
    [0, 1] by the least and largest the tree has seen, 1 the best), one completion per selected path (its actions forced,
    padded with (-1, -1) to the round's deepest path; src = its instance; at most max_candidates per call), and the
    backup of the FP64 objectives w_mk*mk + w_ec*(pt + idle) + w_tt*tt (mtfjsp_mcts_backup).  A node whose child block
    does not fit in the pool stays a leaf.  The decision commits to the root child of the least vmin (the best objective
    through it), ties to the most visits, then the lowest index; the live env steps its action and the root moves there,
    keeping its subtree (no compaction).  A root without children at decision time (its block never fit, or the budget
    never reached it twice) commits to the first action of the decision's best completion -- the base's own action, as
    every path of that decision was the root itself -- and the tree restarts from a fresh root.  Each instance keeps an
    incumbent: the best complete sequence seen (ties keep the earlier), built from the committed prefix, the path and
    the base's actions.  The host reads the round's deepest path once per round.

    With the priority base and simulations >= C + 1 (C the number of candidates, J*M for "all", J for "rule") every root
    child is scored before each decision, so history never increases: the root's own completion begins with the base's
    action, which is a candidate, and that child completes to the same final state, so the least child vmin is at most
    the root's, and the kept subtree carries the value forward.  Below that budget a child nothing reached has vmin =
    +inf and history may increase; the incumbent still never gets worse, so objective <= base_objective always.  With
    the priority base an instance's result depends neither on the batch nor on max_candidates.  With the random base the
    draws are keyed by (seed, decision, round, row of the completion call), so a result depends on the instance's row
    and on how max_candidates splits the rows.
    -> dict: actions [N,S,2] int32 (the incumbents), final4 [S,4], objective [S], history [N+1,S] (history[0] the base's
       completion from the start, history[k+1] the vmin of the child committed at decision k, or the root's for a root
       without children), base_objective [S], completions (completion runs), env_steps (steps they took) and nodes [S]
       (the most pool nodes a tree used at once)."""
    t = np.asarray(instances["t"], dtype=np.float64)
    p = np.asarray(instances["p"], dtype=np.float64)
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    if candidates not in ("all", "rule"):
        raise ValueError("candidates must be 'all' or 'rule'")
    if isinstance(base, str):
        if base != "random":
            raise ValueError("base must be 'random' or an (operation rule, machine rule) pair")
        if candidates == "rule":
            raise ValueError("candidates='rule' needs a rule pair as the base")
        kind = "random"
    else:
        kind = "priority"
    if mask_mode == MASK_ESA:
        raise ValueError("mcts_search supports the FINISHED job mask only: the ESA mask needs state estimates per node")
    if mask_mode != MASK_FINISHED:
        raise ValueError("mask_mode must be MASK_FINISHED")
    if int(simulations) < 1 or int(leaves) < 1 or int(max_nodes) < 1 or max_candidates < 1:
        raise ValueError("simulations, leaves, max_nodes and max_candidates must be >= 1")
    if not (np.isfinite(c) and c >= 0):
        raise ValueError("c must be finite and >= 0")
    L = int(leaves)
    rounds = -(-int(simulations) // L)
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32,
                           mask_mode=mask_mode)
    dev = env.device
    env.load(t, p, np.asarray(instances["transT"]), np.asarray(instances["edge"]))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    key = mach_tab = None
    if kind == "priority":
        k_np, m_np = priority_table(base[0], base[1], t, p, J, M)
        key, mach_tab = torch.as_tensor(k_np, device=dev), torch.as_tensor(m_np, device=dev)
    rule = mach_tab if candidates == "rule" else None
    C = J * M if candidates == "all" else J
    t_dev = torch.as_tensor(t, device=dev)
    tree = mcts_trees(S, max_nodes, dev)
    inst = torch.arange(S, device=dev)
    R = S * L
    src = (torch.arange(R, device=dev) // L).to(torch.int32)
    steps_n = torch.arange(N, device=dev)[:, None]
    env_steps = torch.zeros((), dtype=torch.int64, device=dev)
    bad = torch.zeros((), dtype=torch.bool, device=dev)
    completions = S

    f4, _, fi, ba = env.complete(inst.to(torch.int32), None, base=kind, key=key, mach=mach_tab,
                                 seed=int(np.random.SeedSequence([int(seed), 0]).generate_state(1, dtype=np.uint64)[0]),
                                 mask_mode=mask_mode)
    env_steps += (ba[..., 0] >= 0).sum()
    obj0 = torch.where(fi == -1, _objective(f4, weights), float("inf"))
    inc_obj, inc_f4, inc_act = obj0, f4, ba.clone()
    history = [obj0]
    nodes = tree["count"].clone()
    env.obs(mask_mode)
    acts = torch.full((N, S, 2), -1, dtype=torch.int32, device=dev)
    fresh_tree = mcts_trees(1, 1, dev)
    for k in range(N):
        next_op = torch.where(env.job_mask.bool(), M,
                              env.candidate - torch.arange(J, dtype=torch.int32, device=dev) * M).to(torch.int32)
        dec_obj = torch.full((S,), float("inf"), dtype=torch.float64, device=dev)
        dec_first = torch.full((S, 2), -1, dtype=torch.int32, device=dev)
        for rnd in range(rounds):
            paths, depth, leaf = mcts_select(t_dev, next_op, tree, L, c, rule, N)
            T = int(depth.max())                                              # the one read of the round
            act = paths[:, :T].transpose(0, 1) if T else None
            ds = int(np.random.SeedSequence([int(seed), k + 1, rnd]).generate_state(1, dtype=np.uint64)[0])
            f4 = torch.empty((R, 4), dtype=torch.float64, device=dev)
            fi = torch.empty((R,), dtype=torch.int32, device=dev)
            ba = torch.empty((N, R, 2), dtype=torch.int32, device=dev)
            for c0 in range(0, R, max_candidates):
                c1 = min(R, c0 + max_candidates)
                f4[c0:c1], _, fi[c0:c1], ba[:, c0:c1] = env.complete(
                    src[c0:c1], None if act is None else act[:, c0:c1], base=kind, key=key, mach=mach_tab, seed=ds,
                    mask_mode=mask_mode)
            completions += R
            env_steps += (ba[..., 0] >= 0).sum() + depth.sum()
            ok = (fi == -1) | (fi == depth)
            bad |= ~ok.all()
            obj = torch.where(ok, _objective(f4, weights), float("inf"))
            mcts_backup(tree, leaf, obj)
            nodes = torch.maximum(nodes, tree["count"])
            # the round's best completion per instance: committed prefix, path, base actions
            b_obj, b_l = obj.view(S, L).min(1)
            row = inst * L + b_l
            d = depth[row].long()[None, :]
            pth = paths[row].transpose(0, 1)                                  # [N,S,2]
            via_path = torch.gather(pth, 0, torch.clamp(steps_n - k, 0, N - 1)[..., None].expand(N, S, 2))
            via_base = torch.gather(ba[:, row], 0, torch.clamp(steps_n - k - d, 0, N - 1)[..., None].expand(N, S, 2))
            seq = torch.where((steps_n < k)[..., None], acts,
                              torch.where((steps_n < k + d)[..., None], via_path, via_base))
            better = b_obj < inc_obj
            inc_act = torch.where(better[None, :, None], seq, inc_act)
            inc_f4 = torch.where(better[:, None], f4[row], inc_f4)
            inc_obj = torch.where(better, b_obj, inc_obj)
            dbetter = b_obj < dec_obj
            dec_first = torch.where(dbetter[:, None], seq[k], dec_first)
            dec_obj = torch.where(dbetter, b_obj, dec_obj)
        # commit: the root child of the least vmin, ties to the most visits, then the lowest index
        node, vmin = tree["node"], tree["vmin"]
        root = tree["root"].long()
        fc, nc = node[inst, root, FIRST].long(), node[inst, root, NCHILD].long()
        has = nc > 0
        ci = torch.arange(C, device=dev)[None, :]
        valid = ci < nc[:, None]
        idx = torch.where(valid, fc[:, None] + ci, 0)
        cv = torch.where(valid, vmin[inst[:, None], idx], float("inf"))
        cn = torch.where(valid, node[inst[:, None], idx, VISITS], -1)
        tie = valid & (cv == cv.min(1, keepdim=True)[0])
        cn = torch.where(tie, cn, -1)
        pick = (tie & (cn == cn.max(1, keepdim=True)[0])).long().argmax(1)
        chosen = idx[inst, pick]
        a = torch.where(has[:, None], node[inst, chosen][:, OP:MACH + 1], dec_first)
        history.append(torch.where(has, vmin[inst, chosen], vmin[inst, root]))
        acts[k] = a
        env.step_obs(a[:, 0].contiguous(), a[:, 1].contiguous(), mask_mode)
        # move the root, or restart a tree whose root had no child
        tree["root"] = torch.where(has, chosen, 0).to(torch.int32)
        tree["count"] = torch.where(has, tree["count"], 1).to(torch.int32)
        tree["lohi"] = torch.where(has[:, None], tree["lohi"], fresh_tree["lohi"])
        tree["node"][:, 0] = torch.where(has[:, None], node[:, 0], fresh_tree["node"][:, 0])
        tree["vmin"][:, 0] = torch.where(has, vmin[:, 0], fresh_tree["vmin"][:, 0])
    if bool(bad):
        raise RuntimeError("a completion met an invalid action other than its path's padding")
    out = {"actions": inc_act.cpu().numpy(), "final4": inc_f4.cpu().numpy(), "objective": inc_obj.cpu().numpy(),
           "history": torch.stack(history).cpu().numpy(), "base_objective": obj0.cpu().numpy(),
           "completions": completions, "env_steps": int(env_steps.item()), "nodes": nodes.cpu().numpy()}
    env.close()
    return out
