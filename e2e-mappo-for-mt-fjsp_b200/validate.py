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
