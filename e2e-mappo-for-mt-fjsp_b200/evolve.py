"""NSGA-II over the three targets of a finished schedule (mk, ec = pt + idle, tt; pareto.objectives), on the
environment's whole-episode replay.

A schedule is the complete, valid action sequence a = [(o_s, m_s)], s = 0 .. N-1, of one instance (N = J*M, op o is
operation o % M of job o // M).  The variation operator works on its job-sequence view: position s holds job o_s // M,
and each op keeps its machine apart.  Decoding a job sequence gives position s the op j*M + (the number of earlier
occurrences of j), so every child is complete, in job order, and keeps feasible machines: no repair step.  The operator
is mtfjsp_offspring (csrc/mtfjsp_evolve.cu); `offspring_reference` restates it in numpy draw for draw.

`nsga2` is elitist (mu + lambda) NSGA-II per instance: binary tournaments on (rank, crowding distance), `pop` children by
the operator, replay, non-dominated sorting of parents and children together (mtfjsp_pareto_rank) and the crowding
distance within each front (pareto.crowding_distance) select the next population.  Searching from random individuals
only, it builds a front without any trained policy.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, pareto
from ._lib import _ptr, _stream, check
from .env import BatchedMTFJSPEnv
from .search import _replay_all

_U64 = (1 << 64) - 1


def _offspring_flat(t_dev, M, parents, pair, inst, seed, p_swap, p_mach):
    """mtfjsp_offspring on the kernel's layouts: t_dev [S,N,M] f64, parents [P,N,2] int32, pair [C,2] int32, inst [C]
    int32, all contiguous on one device -> children [C,N,2] int32."""
    S, N = t_dev.shape[0], t_dev.shape[1]
    C, P = pair.shape[0], parents.shape[0]
    children = torch.empty((C, N, 2), dtype=torch.int32, device=t_dev.device)
    if C == 0:
        return children
    if P == 0:  # no parent is read; the library still wants an address
        parents = torch.zeros((1, N, 2), dtype=torch.int32, device=t_dev.device)
    check(_lib.lib().mtfjsp_offspring(_ptr(t_dev), S, N // M, M, _ptr(parents), P, _ptr(pair), _ptr(inst), C,
                                      int(seed) & _U64, float(p_swap), float(p_mach), _ptr(children), _stream()),
          "mtfjsp_offspring")
    return children


def offspring(t, parents, pair, inst, seed=0, p_swap=0.0, p_mach=0.0, device=None):
    """Children of parent sequences (mtfjsp_offspring): [N,C,2] int32 on the device.
    t [S,N,M] processing times (t < 0: infeasible); parents [N,P,2] (op, machine) sequences; pair [C,2] the two parent
    indices of each child, pair[c,0] = -1 for a random child; inst [C] each child's instance.  numpy or torch; the
    device of `parents` if it is a CUDA tensor, else `device` or cuda.

    Child c works on the job-sequence views of its parents.  Its draws are u_k = splitmix64(seed ^ splitmix64(c *
    0x100000001B3 + k * 0x9E3779B97F4A7C15)) >> 11, times 2^-53, a function of (seed, c, k) only; an integer draw below n
    is min(floor(u * n), n - 1).  The draw layout:
      crossover and mutation (pair[c,0] >= 0), J + N + 3 + 2N draws:
        [0, J)            job j is kept when u_j < 0.5 (POX): kept jobs keep parent 1's positions, the other positions
                          take parent 2's non-kept jobs left to right in parent 2's order;
        [J, J+N)          op o's machine is parent 1's when u_{J+o} < 0.5, else parent 2's;
        J+N, J+N+1, J+N+2 when u_{J+N} < p_swap, the job-sequence positions u_{J+N+1} and u_{J+N+2} (below N) swap;
        J+N+3+2o, +1      when u_{J+N+3+2o} < p_mach, op o takes the (u_{J+N+4+2o} below F)-th of its F feasible
                          machines in machine order (it may be the one it had);
      random child (pair[c,0] == -1), 2N draws:
        [1, N)            Fisher-Yates over the job sequence 0..0 1..1 .. (each job M times): for i = N-1 down to 1,
                          position i swaps with position (u_i below i+1);
        [N, 2N)           op o takes the (u_{N+o} below F)-th of its F feasible machines.
    A child with a parent index outside [-1, P) (pair[c,1] outside [0, P) when pair[c,0] >= 0), an instance outside
    [0, S) or a parent holding an op or machine out of range is all -1; the other children are unaffected."""
    dev = parents.device if torch.is_tensor(parents) and parents.is_cuda else torch.device(device or "cuda")
    t_dev = torch.as_tensor(t).to(dev, torch.float64).contiguous()
    if t_dev.dim() != 3:
        raise ValueError("t must have shape [S, N, M]")
    N, M = t_dev.shape[1], t_dev.shape[2]
    par = torch.as_tensor(parents).to(dev, torch.int32)
    if par.dim() != 3 or par.shape[0] != N or par.shape[2] != 2:
        raise ValueError("parents must have shape [%d, P, 2]" % N)
    pr = torch.as_tensor(pair).to(dev, torch.int32).contiguous()
    ic = torch.as_tensor(inst).to(dev, torch.int32).contiguous()
    if pr.dim() != 2 or pr.shape[1] != 2 or tuple(ic.shape) != (pr.shape[0],):
        raise ValueError("pair must have shape [C, 2] and inst [C]")
    out = _offspring_flat(t_dev, M, par.transpose(0, 1).contiguous(), pr, ic, seed, p_swap, p_mach)
    return out.transpose(0, 1)


def _select(f4, pop):
    """Environmental selection of every instance's members f4 [S,K,4] (merged order): the first `pop` by (rank, larger
    crowding distance within the instance's front, merged index).  -> flat indices s*K + k of the survivors [S,pop] in
    that order, and their ranks [S,pop] int32."""
    S, K = f4.shape[0], f4.shape[1]
    dev = f4.device
    obj = pareto.objectives(f4).reshape(S * K, 3)
    rank = pareto.pareto_rank(obj, torch.arange(S + 1, dtype=torch.int64, device=dev) * K, max_len=K)
    r = torch.clamp(rank.long(), 0, K)                                     # a non-finite point (INT32_MAX): last
    inst = torch.arange(S, device=dev).repeat_interleave(K)
    cd = pareto.crowding_distance(obj, inst * (K + 1) + r, S * (K + 1))
    o = torch.sort(-cd, stable=True)[1]                                    # larger distance first, ties by index
    o = o[torch.sort(r[o], stable=True)[1]]
    o = o[torch.sort(inst[o], stable=True)[1]]
    sel = o.view(S, K)[:, :pop]
    return sel, rank[sel]


def _generation_draws(seed, gen, S, pop):
    """Tournament entrants [S,pop,4] int32 (two per parent) and the operator's seed of generation `gen` (0: the start)."""
    state = np.random.SeedSequence([int(seed), int(gen)]).generate_state(2, dtype=np.uint64)
    g = torch.Generator().manual_seed(int(state[0]) & 0x7FFFFFFFFFFFFFFF)
    return torch.randint(0, pop, (S, pop, 4), generator=g, dtype=torch.int32), int(state[1])


def nsga2(instances, actions=None, pop=256, generations=100, p_swap=0.2, p_mach=None, weights=(0.4, 0.4, 0.2),
          left_shift=True, seed=0, max_candidates=65536, device=None):
    """Elitist NSGA-II per instance over (mk, ec, tt) on one env handle of the instances {"t","p","transT","edge"}
    [S,...].

    Start: `actions` ([N,S,2] or [N,K,S,2] integers, numpy or torch: complete valid schedules; None: K = 0) is replayed
    (an invalid start raises ValueError) and filled with pop - K random individuals per instance (mtfjsp_offspring,
    generation 0); a start of more than `pop` members is cut by the selection below.  p_mach=None means 1/N.
    One generation g = 1 .. generations, per instance:
      1. binary tournaments: the population is kept in selection order (rank, larger crowding distance, index), so of
         two entrants the lower index wins.  Entrants come from a torch generator seeded by SeedSequence([seed, g]),
         drawn [S,pop,4] (row s, member i: two tournaments);
      2. `pop` children by mtfjsp_offspring, child s*pop + i from the tournament winners of row (s, i), with p_swap and
         p_mach, under the second word of the same SeedSequence;
      3. the children are replayed from their instance's episode start, at most `max_candidates` per replay call;
      4. parents, then children, are ranked by mtfjsp_pareto_rank;
      5. the crowding distance is taken within each (instance, front) (pareto.crowding_distance);
      6. the first `pop` by (rank, larger crowding distance, merged index) survive, in that order.
    The loop has static sizes and no host synchronisation; the invalid-replay flag is read once at the end (a set flag
    raises RuntimeError).  Every draw is keyed by (instance row, member), so an instance's result depends neither on
    max_candidates nor on the other instances' data; it depends on its row of the batch.
    -> dict of numpy arrays: actions [N,S,pop,2] int32, final4 [S,pop,4], objectives [S,pop,3], rank [S,pop] int32 (in
       the last merged set), ref [S,3] (pareto.reference_point of the start population: the given start and the
       random fill), hypervolume [generations+1, S] (of the rank-0 members in ref, the start population's first), and
       replays, the number of sequences replayed (the start included)."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J, E = N // M, np.asarray(instances["edge"]).shape[1]
    pop, generations = int(pop), int(generations)
    if max_candidates < 1 or generations < 0 or not 1 <= 2 * pop <= pareto.HV_MAX_POINTS:
        raise ValueError("max_candidates must be >= 1, generations >= 0 and 1 <= pop <= %d"
                         % (pareto.HV_MAX_POINTS // 2))
    p_mach = 1.0 / N if p_mach is None else float(p_mach)
    env = BatchedMTFJSPEnv(S, J, M, E, left_shift=left_shift, weights=weights, device=device, obs_dtype=torch.float32)
    dev = env.device
    env.load(*(np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    env.reset(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    t_dev = torch.as_tensor(t, device=dev, dtype=torch.float64).contiguous()

    # the start population: [S,K0,N,2] sequences, K0 = max(K, pop), the given start first
    if actions is None:
        start = torch.zeros((S, 0, N, 2), dtype=torch.int32, device=dev)
    else:
        start = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).to(dev, torch.int32)
        if start.dim() == 3:
            start = start[:, None]
        if start.dim() != 4 or (start.shape[0], start.shape[2], start.shape[3]) != (N, S, 2):
            raise ValueError("actions must have shape [%d, %d, 2] or [%d, K, %d, 2]" % (N, S, N, S))
        start = start.permute(2, 1, 0, 3).contiguous()
    K = start.shape[1]
    if K > pareto.HV_MAX_POINTS:
        raise ValueError("at most %d start sequences per instance" % pareto.HV_MAX_POINTS)
    f4s, bad = _replay_all(env, S * K, lambda a, b: start.view(S * K, N, 2)[a:b].transpose(0, 1),
                           torch.arange(S, device=dev, dtype=torch.int32).repeat_interleave(K), max_candidates)
    if bool(bad):
        raise ValueError("a starting sequence has an invalid action")
    R0 = max(pop - K, 0)
    _, seed0 = _generation_draws(seed, 0, S, pop)
    inst0 = torch.arange(S, device=dev, dtype=torch.int32).repeat_interleave(R0)
    rand = _offspring_flat(t_dev, M, start.view(S * K, N, 2), torch.full((S * R0, 2), -1, dtype=torch.int32, device=dev),
                           inst0, seed0, 0.0, 0.0)
    f4r, bad = _replay_all(env, S * R0, lambda a, b: rand[a:b].transpose(0, 1), inst0, max_candidates)
    K0 = K + R0
    acts = torch.cat((start, rand.view(S, R0, N, 2)), 1)                     # [S,K0,N,2]
    f4 = torch.cat((f4s.view(S, K, 4), f4r.view(S, R0, 4)), 1)               # [S,K0,4]
    replays = S * K0
    ref_np = pareto.reference_point(pareto.objectives(f4).transpose(0, 1).cpu().numpy())
    ref = torch.as_tensor(ref_np, device=dev)

    def survive(acts, f4):
        sel, rank = _select(f4, pop)
        return acts.view(-1, N, 2)[sel.reshape(-1)].view(S, pop, N, 2), f4.view(-1, 4)[sel.reshape(-1)].view(S, pop, 4), rank

    seg_p = torch.arange(S + 1, dtype=torch.int64, device=dev) * pop

    def front_hv(f4, rank):
        o = pareto.objectives(f4).reshape(S * pop, 3)
        o = torch.where((rank.reshape(-1) == 0)[:, None], o, float("nan"))   # other fronts take no part
        return pareto.hypervolume(o, seg_p, ref)

    acts, f4, rank = survive(acts, f4)
    history = [front_hv(f4, rank)]
    inst_c = torch.arange(S, device=dev, dtype=torch.int32).repeat_interleave(pop)
    row = (torch.arange(S, device=dev, dtype=torch.int32) * pop)[:, None]
    for gen in range(1, generations + 1):
        entrants, kseed = _generation_draws(seed, gen, S, pop)
        e = entrants.pin_memory().to(dev, non_blocking=True) if dev.type == "cuda" else entrants.to(dev)
        pair = torch.stack((row + torch.minimum(e[..., 0], e[..., 1]), row + torch.minimum(e[..., 2], e[..., 3])), -1)
        kids = _offspring_flat(t_dev, M, acts.view(S * pop, N, 2), pair.view(S * pop, 2).contiguous(), inst_c, kseed,
                               p_swap, p_mach)
        f4k, badk = _replay_all(env, S * pop, lambda a, b: kids[a:b].transpose(0, 1), inst_c, max_candidates)
        bad = bad | badk
        replays += S * pop
        acts, f4, rank = survive(torch.cat((acts, kids.view(S, pop, N, 2)), 1),
                                 torch.cat((f4, f4k.view(S, pop, 4)), 1))
        history.append(front_hv(f4, rank))
    if bool(bad):
        raise RuntimeError("a child replayed with an invalid action")
    env.close()
    return {"actions": acts.permute(2, 0, 1, 3).cpu().numpy(), "final4": f4.cpu().numpy(),
            "objectives": pareto.objectives(f4).cpu().numpy(), "rank": rank.cpu().numpy(), "ref": ref_np,
            "hypervolume": torch.stack(history).cpu().numpy(), "replays": replays}


# --------------------------------------------------------------------------------------- numpy specification (reference)
def _splitmix64(x):
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def _draws(seed, c, n):
    """u_0 .. u_{n-1} of child c."""
    with np.errstate(over="ignore"):
        k = np.arange(n, dtype=np.uint64)
        x = _splitmix64(np.uint64(int(seed) & _U64) ^ _splitmix64(np.uint64(c) * np.uint64(0x100000001B3)
                                                                  + k * np.uint64(0x9E3779B97F4A7C15)))
    return (x >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def _below(u, n):
    return min(int(u * n), n - 1)


def _nth_feasible(t_row, u):
    feas = np.flatnonzero(t_row >= 0)
    return int(feas[_below(u, len(feas))]) if len(feas) else -1


def offspring_reference(t, parents, pair, inst, seed=0, p_swap=0.0, p_mach=0.0):
    """numpy restatement of mtfjsp_offspring, draw for draw (the layout of `offspring`'s docstring): [N,C,2] int32.
    Arguments as `offspring`, numpy."""
    t = np.asarray(t, dtype=np.float64)
    S, N, M = t.shape
    J = N // M
    par = np.asarray(parents, dtype=np.int64)                              # [N,P,2]
    pair = np.asarray(pair, dtype=np.int64).reshape(-1, 2)
    inst = np.asarray(inst, dtype=np.int64).reshape(-1)
    P, C = par.shape[1], pair.shape[0]
    out = np.full((N, C, 2), -1, dtype=np.int32)

    def in_range(k):
        return ((par[:, k, 0] >= 0) & (par[:, k, 0] < N) & (par[:, k, 1] >= 0) & (par[:, k, 1] < M)).all()

    for c in range(C):
        a, b, s = int(pair[c, 0]), int(pair[c, 1]), int(inst[c])
        if not 0 <= s < S or not -1 <= a < P or (a >= 0 and not 0 <= b < P):
            continue
        if a >= 0 and not (in_range(a) and in_range(b)):
            continue
        if a < 0:
            u = _draws(seed, c, 2 * N)
            x = np.arange(N) // M
            for i in range(N - 1, 0, -1):
                k = _below(u[i], i + 1)
                x[i], x[k] = x[k], x[i]
            mach = np.array([_nth_feasible(t[s, o], u[N + o]) for o in range(N)])
        else:
            u = _draws(seed, c, J + N + 3 + 2 * N)
            p1, p2 = par[:, a], par[:, b]
            m1 = np.empty(N, dtype=np.int64)
            m2 = np.empty(N, dtype=np.int64)
            m1[p1[:, 0]] = p1[:, 1]
            m2[p2[:, 0]] = p2[:, 1]
            kept = u[:J] < 0.5
            j1, j2 = p1[:, 0] // M, p2[:, 0] // M
            x = j1.copy()
            x[~kept[j1]] = j2[~kept[j2]]
            mach = np.where(u[J:J + N] < 0.5, m1, m2)
            for o in np.flatnonzero(u[J + N + 3:J + 3 * N + 3:2] < p_mach):
                r = _nth_feasible(t[s, o], u[J + N + 4 + 2 * o])
                if r >= 0:
                    mach[o] = r
            if u[J + N] < p_swap:
                i, k = _below(u[J + N + 1], N), _below(u[J + N + 2], N)
                x[i], x[k] = x[k], x[i]
        order = np.argsort(x, kind="stable")
        occ = np.empty(N, dtype=np.int64)
        occ[order] = np.arange(N) - np.searchsorted(x[order], x[order])   # earlier occurrences of the same job
        op = x * M + occ
        out[:, c, 0] = op
        out[:, c, 1] = mach[op]
    return out
