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

`pareto_local_search` walks the same neighbourhood without a weighted sum: it keeps an archive of mutually
non-dominated schedules per instance over the three targets (pareto.py) and expands it until no member is left
unexplored.
"""
from __future__ import annotations

import numpy as np
import torch

from . import pareto
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
