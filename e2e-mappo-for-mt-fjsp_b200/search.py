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
"""
from __future__ import annotations

import numpy as np
import torch

from .env import BatchedMTFJSPEnv
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
    after each round, the start first; never increasing), accepted [rounds_run, S] bool."""
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
    inst_ids = torch.arange(S, device=dev)
    for rnd in range(int(rounds)):
        moves = neighbour_moves(cur, t_dev, max_neighbours, seed, rnd)
        R = moves.shape[0]
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
            "accepted": (torch.stack(accepted) if accepted else torch.zeros((0, S), dtype=torch.bool)).cpu().numpy()}
