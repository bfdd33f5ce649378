"""Batched priority-dispatching-rule (PDR) rollouts on the device (SURVEY.md 8 f-4).

The reference evaluates 6 operation rules x 2 machine rules one instance at a time through the networkx env
(tester/pdrs.py:611-839, test_all.py:484-503; 0.14-0.2 s per 36-step episode).  The rules below are static orders
computed from the instance tables, so a whole instance set is scheduled in J*M env-kernel launches.

Operation rules (tester/pdrs.py): FIFO (:123-125), LWKR_T / MWKR_T (:162-224, data_type "mean"),
LWKR_PT / MWKR_PT (:226-288).  Machine rules: SPT (:46-52), SEC (:55-62).  Rollouts run WITHOUT left shift, as the
reference's do (tester/pdrs.py:669).  `evaluate_rules` reproduces the shipped result rows
results/test_results/Real_{MK,PT,TT,IT}_J6_M6_E2_Seed3_Weight442.csv bit for bit (tests/test_rules.py).

State-dependent rules, on the environment's one-step lookahead (BatchedMTFJSPEnv.peek):
LWKR_IT / MWKR_IT (tester/pdrs.py:465-540, LWKR_IT_o_jointActor with type "min" / "max") pick, among the jobs with an
unscheduled op, the one whose candidate op on the machine rule's machine adds the least / most idle time: the largest /
smallest r_idle = previous - new idle time.  The reference replays the whole chosen prefix for every candidate of every
decision and left these rules out of its test table; here one peek per decision answers for every job.  Deviation: the
reference breaks ties with random.choice, here the lowest job index wins, as in the static rules above.
GREEDY_R is this project's own joint baseline, not the reference's: at every step the valid (candidate op, machine)
pair with the largest step reward r, ties to the lowest j*M + m.
"""
from __future__ import annotations

import numpy as np
import torch

from .env import BatchedMTFJSPEnv

OP_RULES = ("FIFO", "LWKR_T", "LWKR_PT", "MWKR_T", "MWKR_PT")
MACHINE_RULES = ("SPT", "SEC")
LOOKAHEAD_RULES = ("LWKR_IT", "MWKR_IT")
JOINT_RULES = ("GREEDY_R",)


def machine_rule(name, t, p):
    """[S,N,M] tables -> [S,N] machine of every op.  SPT: shortest feasible time; SEC: smallest feasible t*|p|."""
    if name == "SPT":
        v = np.where(t < 0, np.inf, t)
    elif name == "SEC":
        e = t * np.abs(p)
        v = np.where(e < 0, np.inf, e)
    else:
        raise ValueError(name)
    return np.argmin(v, axis=-1)


def _row_mean_positive(x):
    """python-order mean of the positive entries of each row: sum(left to right) / count (pdrs.py:171-176)."""
    S, N, M = x.shape
    acc = np.zeros((S, N))
    cnt = np.zeros((S, N))
    for m in range(M):
        pos = x[:, :, m] > 0
        acc = np.where(pos, acc + x[:, :, m], acc)
        cnt += pos
    return np.where(cnt > 0, acc / np.maximum(cnt, 1), 0.0)


def _op_rule_walk(name, t, p, n_job, n_machine):
    """The op rule's loop (pdrs.py:186-197) -> ([S,N] op order, [S,N] f64 priority key of every op).
    The key of op j*M + k is the rule's value of job j when that op is next: refer[j] after k subtractions (LWKR), its
    negation (MWKR), the op index (FIFO); +inf for an op the loop never reaches because its job was finished by
    refer == 0.  Taking, at every step, the job whose next op has the smallest key, ties to the lowest job, gives the
    order back."""
    S, N, M = t.shape
    J = n_job
    if name == "FIFO":
        return np.tile(np.arange(N), (S, 1)), np.tile(np.arange(N, dtype=np.float64), (S, 1))
    least = name.startswith("LWKR")
    if name.endswith("_PT"):
        sel = _row_mean_positive(t * np.abs(p))
    else:
        sel = _row_mean_positive(t)
    tn = sel.reshape(S, J, M)
    refer = np.sum(tn, axis=2)                      # np.sum over the job's ops (pairwise order = numpy's)
    nxt = np.zeros((S, J), dtype=np.int64)
    order = np.zeros((S, N), dtype=np.int64)
    key = np.full((S, N), np.inf)
    ar = np.arange(S)
    for s in range(N):                              # pdrs.py:186-197
        j = np.argmin(refer, axis=1) if least else np.argmax(refer, axis=1)
        order[:, s] = j * M + nxt[ar, j]
        key[ar, order[:, s]] = refer[ar, j] if least else -refer[ar, j]
        refer[ar, j] = refer[ar, j] - tn[ar, j, nxt[ar, j]]
        nxt[ar, j] += 1
        fin = (refer[ar, j] == 0) | (nxt[ar, j] > M - 1)
        refer[ar, j] = np.where(fin, np.inf if least else -np.inf, refer[ar, j])
    return order, key


def op_rule(name, t, p, n_job, n_machine):
    """-> [S,N] op order (0-based op ids, position s = the op scheduled at step s)."""
    return _op_rule_walk(name, t, p, n_job, n_machine)[0]


def priority_table(op_rule_name, machine_rule_name, t, p, n_job, n_machine):
    """A static rule pair as priority tables for the device completion (BatchedMTFJSPEnv.complete, base "priority"):
    key [S,N] f64 and mach [S,N] int32.  From the reset state, with the FINISHED job mask, the priority completion
    schedules exactly op_rule's order on machine_rule's machines, as evaluate_rules steps them."""
    t = np.asarray(t, dtype=np.float64)
    p = np.asarray(p, dtype=np.float64)
    key = _op_rule_walk(op_rule_name, t, p, n_job, n_machine)[1]
    return key, machine_rule(machine_rule_name, t, p).astype(np.int32)


def lookahead_choice(name, r_idle, invalid):
    """The LWKR_IT / MWKR_IT decision: [B,J] r_idle of every job's candidate (the machine rule's machine) and [B,J]
    invalid flags -> [B,1] int64 chosen job.  LWKR_IT (the reference's "min") takes the largest r_idle = previous - new
    idle time (<= 0 without left shift), MWKR_IT ("max") the smallest; ties go to the lowest job index."""
    if name == "LWKR_IT":
        return torch.where(invalid == 0, r_idle, -torch.inf).argmax(dim=1, keepdim=True)
    if name == "MWKR_IT":
        return torch.where(invalid == 0, r_idle, torch.inf).argmin(dim=1, keepdim=True)
    raise ValueError(name)


def lookahead_rollout(env, name, machines):
    """Runs LWKR_IT or MWKR_IT on a freshly reset env: machines [B,N] integer tensor (the machine rule's machine of every
    op).  N decisions on the device, no host synchronisation.  Returns the actions [N,B,2] int32 (op, machine)."""
    machines = machines.to(device=env.device, dtype=torch.int32)
    acts = []
    for _ in range(env.N):
        cand = env.candidate_ops()                                        # [B,J]
        mch = torch.gather(machines, 1, cand.long())
        r5, inv = env.peek(cand, mch)
        j = lookahead_choice(name, r5[..., 2], inv)
        a = torch.cat((torch.gather(cand, 1, j), torch.gather(mch, 1, j)), dim=1)
        env.step(a[:, 0].contiguous(), a[:, 1].contiguous())
        acts.append(a)
    return torch.stack(acts)


def greedy_reward_rollout(env):
    """GREEDY_R on a freshly reset env: at every step the valid (candidate op, machine) pair with the largest step
    reward r, ties to the lowest j*M + m.  N decisions on the device, no host synchronisation.  Returns the actions
    [N,B,2] int32 (op, machine)."""
    B, J, M = env.B, env.J, env.M
    acts = []
    for _ in range(env.N):
        cand = env.candidate_ops()
        op = cand.unsqueeze(2).expand(B, J, M).reshape(B, J * M)
        mach = torch.arange(M, dtype=torch.int32, device=env.device).repeat(J).expand(B, J * M)
        r5, inv = env.peek(op, mach)
        k = torch.where(inv == 0, r5[..., 0], -torch.inf).argmax(dim=1, keepdim=True)
        a = torch.cat((torch.gather(cand, 1, k // M), (k % M).to(torch.int32)), dim=1)
        env.step(a[:, 0].contiguous(), a[:, 1].contiguous())
        acts.append(a)
    return torch.stack(acts)


def evaluate_rules(t, p, transT, edge, n_job, n_machine, n_edge, op_rules=OP_RULES, machine_rules=MACHINE_RULES,
                   weights=(0.4, 0.4, 0.2), device=None, joint_rules=()):
    """Schedules every instance with every (operation rule, machine rule) pair, then with every joint rule.
    op_rules: names from OP_RULES and LOOKAHEAD_RULES; joint_rules: names from JOINT_RULES (not crossed with the machine
    rules; row name = the rule's name).
    Returns dict: names [R], costs [R,S,4] = (makespan, processing energy / N, transport time, idle time) and
    objective [R,S] = w_mk*mk + w_ec*(pt + idle) + w_tt*tt (trainer/validate.py:283)."""
    t = np.asarray(t, dtype=np.float64)
    p = np.asarray(p, dtype=np.float64)
    S, N, M = t.shape
    env = BatchedMTFJSPEnv(S, n_job, n_machine, n_edge, left_shift=False, weights=weights, device=device,
                           obs_dtype=torch.float32)
    env.load(t, p, transT, edge)
    env.scaler_init()
    w = torch.tensor(np.tile(np.asarray(weights, dtype=np.float64), (S, 1)))
    names, costs = [], []
    ar = np.arange(S)

    def finish(name):
        if int(env.invalid.sum().item()) != 0 or int(env.done.sum().item()) != S:
            raise RuntimeError("rule %s produced an invalid schedule" % name)
        names.append(name)
        costs.append(env.costs().cpu().numpy())

    for orule in op_rules:
        order = None if orule in LOOKAHEAD_RULES else op_rule(orule, t, p, n_job, n_machine)
        for mrule in machine_rules:
            mch = machine_rule(mrule, t, p)
            env.reset(w)
            if order is None:
                lookahead_rollout(env, orule, torch.as_tensor(mch.astype(np.int32)).to(env.device))
            else:
                ops_dev = torch.as_tensor(order.T.astype(np.int32).copy()).to(env.device)                      # [N,S]
                mch_dev = torch.as_tensor(mch[ar[:, None], order].T.astype(np.int32).copy()).to(env.device)    # [N,S]
                for s in range(N):
                    env.step(ops_dev[s], mch_dev[s])
            finish("%s+%s" % (orule, mrule))
    for jrule in joint_rules:
        if jrule not in JOINT_RULES:
            raise ValueError(jrule)
        env.reset(w)
        greedy_reward_rollout(env)
        finish(jrule)
    costs = np.stack(costs)
    obj = weights[0] * costs[..., 0] + weights[1] * (costs[..., 1] + costs[..., 3]) + weights[2] * costs[..., 2]
    return dict(names=names, costs=costs, objective=obj)
