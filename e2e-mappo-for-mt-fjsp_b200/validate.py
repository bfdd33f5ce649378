"""Batched greedy and sampled validation of a trained policy (SURVEY.md 8 f-4; reference: trainer/validate.py:60-297, one
instance at a time, batch 1, env on the CPU and both actors on the GPU; driven 100 times per evaluation by
Run.py:672-814 and test_all.py:260-334).

Here the S instances are one env batch on the device and every rollout step is one forward of each actor over all of
them.  The reference's modules are never put in eval mode, so a batch-1 validation normalises every BatchNorm with the
statistics of that ONE instance's rows (SURVEY.md 3.3); `per_instance_batchnorm=True` keeps exactly that by giving each
instance its own BatchNorm group, which is what makes the results comparable with the reference's (and with the
shipped result CSV rows `PPO-G` / `new12800`).  With False the statistics run over the whole batch (the training-rollout
convention at large env batches).
"""
from __future__ import annotations

import numpy as np
import torch

from .encoder import select
from .env import MASK_ESA, BatchedMTFJSPEnv


def load_actor_state_dicts(npz_path_or_dict, tag):
    """(operation-actor state_dict, machine-actor state_dict) stored as `<tag>/op/<key>` / `<tag>/mch/<key>` arrays
    (tests/golden/policy_golden.npz holds the reference's shipped J6M6E2 checkpoints in that form)."""
    g = np.load(npz_path_or_dict) if isinstance(npz_path_or_dict, str) else npz_path_or_dict
    pick = lambda part: {k.split("/", 2)[2]: torch.as_tensor(g[k]) for k in g.files if k.startswith("%s/%s/" % (tag, part))}
    return pick("op"), pick("mch")


def load_checkpoint(job_pth, mch_pth, n_job, n_machine, precision="fp32", device=None, hidden=128):
    """(JobActor, MachineActor) from two `torch.save`d state_dicts with the reference's key names: the
    `PPO_job_actor_*.pth` / `PPO_machine_actor_*.pth` files `train.Trainer` writes, or the reference's own checkpoints
    (Run.py:773-814).  The pair plugs straight into `greedy_validate` / `sampled_validate`."""
    from .encoder import JobActor, MachineActor

    ld = lambda f: torch.load(f, map_location="cpu", weights_only=True)
    return (JobActor(ld(job_pth), n_job, n_machine, hidden=hidden, device=device, precision=precision),
            MachineActor(ld(mch_pth), n_machine, hidden=hidden, device=device, precision=precision))


def read_mip_csv(path):
    """The MIP result CSV of the reference's solver runs (tester/Solver_seed*/MO_FJSP_MIP_result_(...).csv, parsed as
    trainer/validate.py:14-58 does): a header row, then one row per instance of runtime, best_objective, Makespan,
    MachineEC, MachineIdleT, TransEC -> dict of [S] float64 arrays under those names."""
    import csv

    with open(path, newline="") as f:
        rows = list(csv.reader(f))
    names = ("runtime", "best_objective", "Makespan", "MachineEC", "MachineIdleT", "TransEC")
    data = np.array([[float(v) for v in r] for r in rows[1:] if r], dtype=np.float64).reshape(-1, len(names))
    return {n: data[:, i] for i, n in enumerate(names)}


def mip_gaps(final4, mip, weights=(0.4, 0.4, 0.2)):
    """Relative gaps to the MIP solutions (Run.py:708-716): per instance (cost - mip) / mip of makespan, processing
    energy, transport time and idle time [S,4], and their weighted sum w_mk g_mk + w_ec (g_pt + g_idle) + w_tt g_tt [S]."""
    ref = np.stack((mip["Makespan"], mip["MachineEC"], mip["TransEC"], mip["MachineIdleT"]), axis=-1)[: len(final4)]
    g = (np.asarray(final4) - ref) / ref
    return g, _objective(g, weights)


def _objective(final4, weights):
    w = weights
    return w[0] * final4[..., 0] + w[1] * (final4[..., 1] + final4[..., 3]) + w[2] * final4[..., 2]


def _rollout_chunks(job_actor, machine_actor, instances, weights, left_shift, per_instance_batchnorm, chunk, acts, choose):
    """The rollout loop both validations share: every env of a chunk one step per actor forward, to completion.
    choose(kind, prob_or_scores, mask, cand, chunk_index) -> action index [B] picks the job (kind 0) or machine (kind 1);
    it gets the masked probabilities from `choose.logits = False`, the unmasked scores otherwise.
    -> final4 [S,4], cumulative rewards [S,5]; acts [N,S,2] (or None) receives the actions."""
    t = np.asarray(instances["t"])
    S, N, M = t.shape
    J = N // M
    E = np.asarray(instances["edge"]).shape[1]
    final4 = np.zeros((S, 4))
    cum = np.zeros((S, 5))
    env = None
    for ci, s0 in enumerate(range(0, S, chunk)):
        s1 = min(S, s0 + chunk)
        B = s1 - s0
        if env is None or env.B != B:
            env = BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, weights=weights, obs_dtype=torch.float32,
                                   mask_mode=MASK_ESA)
        env.load(*(np.asarray(instances[k])[s0:s1] for k in ("t", "p", "transT", "edge")))
        env.scaler_init()
        env.reset(np.tile(np.asarray(weights, dtype=np.float64), (B, 1)))
        env.obs(MASK_ESA)
        groups = B if per_instance_batchnorm else 1
        h_mch = None
        tot = torch.zeros((B, 5), dtype=torch.float64, device=env.device)
        with torch.no_grad():
            for step in range(N):
                p, pooled, _ = job_actor.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, h_mch, env.job_mask,
                                                  groups=groups, return_logits=choose.logits)
                a = choose(0, p, env.job_mask, env.candidate, ci)
                env.op.copy_(env.candidate.long().gather(1, a.unsqueeze(-1)).squeeze(-1).to(torch.int32))
                m1, mmask = env.mfea1(env.op)
                mp, h_mch, _ = machine_actor.forward(m1, env.mach_fea, pooled, mmask, groups=groups, return_logits=choose.logits)
                env.mach.copy_(choose(1, mp, mmask, None, ci).to(torch.int32))
                if acts is not None:
                    acts[step, s0:s1, 0] = env.op.cpu().numpy(); acts[step, s0:s1, 1] = env.mach.cpu().numpy()
                env.step_obs(env.op, env.mach, MASK_ESA)
                tot += env.reward5
        assert bool(env.done.all()) and not bool(env.invalid.any())
        final4[s0:s1] = env.costs().cpu().numpy()
        cum[s0:s1] = tot.cpu().numpy()
    return final4, cum


def _greedy_choice(kind, prob, mask, cand, ci):
    return prob.argmax(dim=-1)


_greedy_choice.logits = False


def greedy_validate(job_actor, machine_actor, instances, weights=(0.4, 0.4, 0.2), left_shift=True,
                    per_instance_batchnorm=True, chunk=None, return_actions=False):
    """Greedy rollout of every instance of `instances` ({"t","p","transT","edge"} arrays, [S,...]) to completion.

    -> dict: final4 [S,4] f64 = (makespan, processing energy / N, transport time, idle time) read after `done`
             (validate.py:273-277), objective [S] = w_mk * mk + w_ec * (pt + idle) + w_tt * tt (validate.py:283),
             cumulative rewards [S,5] (validate.py:248-252) and optionally the action sequence [N,S,2].
    Reward weights are the fixed evaluation weights (`reset(Random_weight_type="eval")`, validate.py:142); job mask =
    the ESA rule (`Eval_esa_update_...`, algorithm/ppo_algorithm.py:321-417); both actors take the arg-max
    (agent_func.py:41-51, 65-73; ties resolve to the lowest index as torch.max / torch.argmax do).
    chunk: envs per batch.  The default is 1 for a tf32 job actor with per_instance_batchnorm (one instance per batch, as
    before the grouped tcgen05 encoder existed) and all S otherwise; an explicit chunk > 1 runs the tf32 job actor with one
    BatchNorm group per instance, and every instance's result is the same bits as with chunk=1 (grouped statistics are
    summed in a fixed per-env order)."""
    t = np.asarray(instances["t"])
    S, N = t.shape[0], t.shape[1]
    tf32_job = getattr(job_actor, "precision", "fp32") == "tf32"
    if chunk is None:
        chunk = 1 if (tf32_job and per_instance_batchnorm) else S
    acts = np.zeros((N, S, 2), dtype=np.int32) if return_actions else None
    final4, cum = _rollout_chunks(job_actor, machine_actor, instances, weights, left_shift, per_instance_batchnorm, chunk, acts,
                                  _greedy_choice)
    out = {"final4": final4, "objective": _objective(final4, weights), "cumulative_rewards": cum}
    if acts is not None:
        out["actions"] = acts
    return out


class _SampledChoice:
    """Draws of both actors from the masked softmax (agent_func.py:22-63 with greedy=False): the one-launch selection
    kernel (encoder.select, stream ids 0 / 1, a device step counter) keyed by the chunk's seed, or torch.multinomial on a
    generator seeded the same way where J or M exceeds the kernel's 32 lanes."""

    def __init__(self, seed, J, M, device):
        self.seed = seed
        self.logits = J <= 32 and M <= 32
        self.counter = torch.zeros(1, dtype=torch.int64, device=device)
        self.gen = torch.Generator(device=device)
        self.ci = -1

    def chunk_seed(self, ci):
        return int(np.random.SeedSequence([self.seed, ci]).generate_state(2, dtype=np.uint64)[0])

    def __call__(self, kind, p, mask, cand, ci):
        if ci != self.ci:
            self.ci = ci
            self.counter.zero_()
            self.gen.manual_seed(self.chunk_seed(ci) & 0x7FFFFFFFFFFFFFFF)
        if not self.logits:
            return torch.multinomial(p, 1, generator=self.gen).squeeze(-1)
        _, a, _, _ = select(p, mask, None, 1.0, False, (self.chunk_seed(ci), self.counter), kind)
        if kind == 1:
            self.counter.add_(1)
        return a


def sampled_validate(job_actor, machine_actor, instances, samples, seed=0, weights=(0.4, 0.4, 0.2), left_shift=True,
                     per_instance_batchnorm=True, max_envs=32768, return_actions=False):
    """K = `samples` sampled rollouts of each of the S instances (test_all.py's PPO-S row: `greedy=False`, one
    Categorical draw per actor per step), all in batches on the device, and the best of them per instance.

    Env k * S + s rolls out instance s; the envs run in chunks of at most `max_envs` (which also keeps the tf32 machine
    actor's per-instance BatchNorm under its 65,535 groups per call); chunk c draws with a seed derived from (seed, c), so
    the draws are a function of (seed, max_envs).  With per_instance_batchnorm every env is its own BatchNorm group, as in
    the reference's one-instance-at-a-time test rollouts.
    -> dict: final4 [K,S,4], objective [K,S], cumulative_rewards [K,S,5], best_index [S] (the lowest k on ties),
             best_final4 [S,4], best_objective [S] and, with return_actions, actions [N,K,S,2] and best_actions [N,S,2]."""
    inst = {k: np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")}
    S, N, M = inst["t"].shape
    K = int(samples)
    if K < 1 or max_envs < 1:
        raise ValueError("samples and max_envs must be >= 1")
    rep = {k: np.tile(v, (K,) + (1,) * (v.ndim - 1)) for k, v in inst.items()}
    choose = _SampledChoice(seed, N // M, M, job_actor.device)
    acts = np.zeros((N, K * S, 2), dtype=np.int32) if return_actions else None
    final4, cum = _rollout_chunks(job_actor, machine_actor, rep, weights, left_shift, per_instance_batchnorm, max_envs, acts,
                                  choose)
    final4, cum = final4.reshape(K, S, 4), cum.reshape(K, S, 5)
    obj = _objective(final4, weights)
    best = np.argmin(obj, axis=0)
    cols = np.arange(S)
    out = {"final4": final4, "objective": obj, "cumulative_rewards": cum, "best_index": best,
           "best_final4": final4[best, cols], "best_objective": obj[best, cols]}
    if acts is not None:
        out["actions"] = acts.reshape(N, K, S, 2)
        out["best_actions"] = acts[:, best * S + cols]
    return out


# per-call BatchNorm group limit of the per-group paths (mtfjsp_enc_bn_fwd's grid.y)
_MAX_GROUPS = 65535


def beam_select(score, width):
    """One beam step's selection.  score [S, C] f64: the children of an instance in flat order (w * J + j) * M + m, -inf for
    the impossible ones.  Children rank by (score descending, flat index ascending) and slot w takes the child ranked w; a
    slot whose child scores -inf is dead and takes the rank-0 child instead (so that every env steps validly).
    -> child [S, width] int64 flat index, slot score [S, width] f64 (-inf for a dead slot), alive [S, width] bool."""
    val, order = torch.sort(score, dim=1, descending=True, stable=True)
    val, order = val[:, :width], order[:, :width]
    alive = val > float("-inf")
    return torch.where(alive, order, order[:, :1]), val, alive


def _beam_chunk(job_actor, machine_actor, inst, W, weights, left_shift, per_instance_batchnorm, envs, want_actions):
    """Beam search over one chunk of S instances on the env pair `envs` (two handles of S * W envs, env s * W + w).
    -> final4 [S,W,4], log_prob [S,W], actions [N,S*W,2] (or None), all on the device."""
    S, N, M = inst["t"].shape
    J = N // M
    B = S * W
    A, Bn = envs
    A.load(*(np.repeat(inst[k], W, axis=0) for k in ("t", "p", "transT", "edge")))
    A.scaler_init()
    A.reset(np.tile(np.asarray(weights, dtype=np.float64), (B, 1)))
    A.obs(MASK_ESA)
    dev = A.device
    ninf = float("-inf")
    score = torch.full((S, W), ninf, dtype=torch.float64, device=dev)
    score[:, 0] = 0.0
    job_groups, mach_groups = (B, B * J) if per_instance_batchnorm else (1, 1)
    base = (torch.arange(S, device=dev) * W).unsqueeze(1)
    parents = torch.empty((N, B), dtype=torch.int64, device=dev) if want_actions else None
    acts = torch.empty((N, B, 2), dtype=torch.int32, device=dev) if want_actions else None
    h_mch = None
    with torch.no_grad():
        for step in range(N):
            pj, pooled, _ = job_actor.evaluate(A.task_fea, A.adj_w, A.adj_src, A.candidate, h_mch, A.job_mask, groups=job_groups)
            # the (env, job) children: candidate-machine features of each job's candidate op, child = env * J + j
            f1, mm = [], []
            for j in range(J):
                a, b = A.mfea1(A.candidate[:, j].contiguous())
                f1.append(a.clone())
                mm.append(b.clone())
            f1 = torch.stack(f1, 1).view(B * J, M, -1)
            mm = torch.stack(mm, 1).view(B * J, M)
            pm, hm, _ = machine_actor.forward(f1, A.mach_fea.repeat_interleave(J, 0), pooled.repeat_interleave(J, 0), mm,
                                              groups=mach_groups)
            child = (score.reshape(B, 1, 1) + torch.log(pj).double().reshape(B, J, 1)) + torch.log(pm).double().reshape(B, J, M)
            bad = A.job_mask.bool().reshape(B, J, 1) | mm.bool().reshape(B, J, M)
            child = torch.where(bad, ninf, child)
            pick, score, _ = beam_select(child.view(S, W * J * M), W)
            parent = (base + pick // (J * M)).view(-1)
            job = ((pick // M) % J).view(-1)
            Bn.gather_from(A, parent)
            Bn.op.copy_(Bn.candidate.gather(1, job.unsqueeze(1)).squeeze(1))
            Bn.mach.copy_((pick % M).view(-1))
            h_mch = hm.index_select(0, parent * J + job)
            if want_actions:
                parents[step] = parent
                acts[step, :, 0] = Bn.op
                acts[step, :, 1] = Bn.mach
            Bn.step_obs(Bn.op, Bn.mach, MASK_ESA)
            A, Bn = Bn, A
    if not (bool(A.done.all()) and not bool(A.invalid.any())):
        raise RuntimeError("beam search ended with an unfinished or invalid env")
    final4 = A.costs().view(S, W, 4)
    actions = None
    if want_actions:  # follow every final slot's parents back to the start
        actions = torch.empty_like(acts)
        cur = torch.arange(B, device=dev)
        for step in range(N - 1, -1, -1):
            actions[step] = acts[step].index_select(0, cur)
            cur = parents[step].index_select(0, cur)
    return final4, score, actions


def beam_validate(job_actor, machine_actor, instances, width, weights=(0.4, 0.4, 0.2), left_shift=True,
                  per_instance_batchnorm=True, max_envs=32768, return_actions=False):
    """Deterministic beam search of width W = `width` over joint (job, machine) actions for every instance of `instances`
    ({"t","p","transT","edge"} arrays, [S,...]), on the same actor pairs, precisions and BatchNorm semantics as
    `greedy_validate`.

    Each instance keeps W partial schedules (slots; slot 0 starts live, the others dead at score -inf).  Per step the job
    actor runs on every slot's env, and the machine actor on every (slot, job) child -- with per_instance_batchnorm each
    child is its own BatchNorm group, as a batch-1 validation of that env would be.  A (slot, job, machine) child scores
    parent + log p_job + log p_mach (torch.log of the FP32 probabilities greedy arg-maxes, summed in FP64; masked jobs and
    infeasible machines -inf), and the W best children of the instance become its next slots (`beam_select`: ties to the
    lowest flat index (w * J + j) * M + m; a slot without a finite child is dead and copies the best one).  The envs of the
    chosen parents are copied into a second env batch (`BatchedMTFJSPEnv.gather_from`) and stepped there; the two batches
    swap roles every step.  Instances run in chunks of at most `max_envs` envs (and of at most 65,535 children, the
    per-group BatchNorm limit of one machine-actor call).  With per_instance_batchnorm and tf32 actors an instance's
    result does not depend on the chunking or on the other instances.
    per_instance_batchnorm=False gives each actor call one BatchNorm group over its whole batch, as greedy_validate does,
    but the batch here is not greedy's: the job actor's statistics run over the S_chunk * W slot envs, dead slots (copies
    of their instance's best child) included, and the machine actor's over all S_chunk * W * J (slot, job) children, those
    of masked and finished jobs included.  The result then depends on W, on `max_envs` and on the other instances of the
    chunk; it is not the whole-batch greedy semantics at W = 1 either.
    -> dict: final4 [W,S,4], objective [W,S], log_prob [W,S] (the slot's score), alive [W,S], best_index [S] (the live
             slot of the lowest objective, lowest w on ties), best_final4 [S,4], best_objective [S] and, with
             return_actions, actions [N,W,S,2] (op, machine) and best_actions [N,S,2]."""
    inst = {k: np.asarray(instances[k]) for k in ("t", "p", "transT", "edge")}
    S, N, M = inst["t"].shape
    J, E = N // M, inst["edge"].shape[1]
    W = int(width)
    if W < 1 or max_envs < W:
        raise ValueError("width must be >= 1 and max_envs >= width")
    if W * J > _MAX_GROUPS:
        raise ValueError("width * J = %d children per instance exceed the %d BatchNorm groups of one machine-actor call"
                         % (W * J, _MAX_GROUPS))
    chunk = max(1, min(max_envs // W, _MAX_GROUPS // (W * J)))
    final4 = np.zeros((W, S, 4))
    log_prob = np.zeros((W, S))
    acts = np.zeros((N, W, S, 2), dtype=np.int32) if return_actions else None
    envs = None
    for s0 in range(0, S, chunk):
        s1 = min(S, s0 + chunk)
        B = (s1 - s0) * W
        if envs is None or envs[0].B != B:
            envs = tuple(BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, weights=weights, obs_dtype=torch.float32,
                                          mask_mode=MASK_ESA) for _ in range(2))
        f4, lp, ac = _beam_chunk(job_actor, machine_actor, {k: v[s0:s1] for k, v in inst.items()}, W, weights, left_shift,
                                 per_instance_batchnorm, envs, return_actions)
        final4[:, s0:s1] = f4.transpose(0, 1).cpu().numpy()
        log_prob[:, s0:s1] = lp.t().cpu().numpy()
        if acts is not None:
            acts[:, :, s0:s1] = ac.view(N, s1 - s0, W, 2).transpose(1, 2).cpu().numpy()
    obj = _objective(final4, weights)
    alive = log_prob > -np.inf
    best = np.argmin(np.where(alive, obj, np.inf), axis=0)
    cols = np.arange(S)
    out = {"final4": final4, "objective": obj, "log_prob": log_prob, "alive": alive, "best_index": best,
           "best_final4": final4[best, cols], "best_objective": obj[best, cols]}
    if acts is not None:
        out["actions"] = acts
        out["best_actions"] = acts[:, best, cols]
    return out
