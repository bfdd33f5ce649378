"""Batched MAPPO update on the device (SURVEY.md 8 f-3).

Reference: PPOAlgorithm.global_update_JointActions_GAT_selfCritic (algorithm/ppo_algorithm.py:539-1124) and the
rollout bookkeeping that feeds it (Run.py:290-545, trainer/replaybuffer.py:18-204).

What changes against the reference, and what does not:

* The reference re-runs the three networks ONE BUFFERED STEP AT A TIME inside every minibatch (python loops at
  ppo_algorithm.py:632-659 and :739-775: mini_bs forward passes of B envs each).  Here a minibatch is ONE forward
  over [mini_bs * B] graphs.  The two things that made the loop look sequential are handled explicitly:
    - BatchNorm batch statistics are per buffered step -> `groups = mini_bs` in encoder._bn_train;
    - the job actor of item i receives the machine embedding of item i-1 of the (shuffled) minibatch, item 0 the
      learned `_input` vector (:746 `h_mch_pooled`).  That embedding depends only on item i-1's machine features, so
      all machine trunks are evaluated first and handed on shifted by one.
  Losses, clipping, optimiser steps and their order are the reference's, line for line (cited below).
* Observations are the env's native ones: F32 features and the ELL adjacency (10 bytes per node) instead of two
  dense [steps, B, N, N] float64 adjacencies; the aggregation forward / backward are the hand-written kernels of
  csrc/mtfjsp_encoder.cu, GAE is csrc `gae4_kernel`; the dense layers run on library FP32 GEMMs under autograd.
* Data-parallel training (SURVEY.md 8e): every rank updates on its own env slice, gradients are averaged with one
  NCCL allreduce per backward pass, advantage statistics are summed across ranks (buffer.gae4).  BatchNorm statistics
  stay local to the rank (the reference's statistics are per B-env batch as well).
"""
from __future__ import annotations

from dataclasses import dataclass

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch.distributions import Categorical

from . import encoder as _enc
from .buffer import RolloutBuffer, gae4
from .rollout import nvtx_range


@dataclass
class PPOConfig:
    """Defaults of the reference's parameters.py:77-97."""
    lr: float = 1e-3
    lr_eps: float = 1e-5
    use_lr_decay: bool = False
    decay_step_size: int = 20
    decay_ratio: float = 0.96
    gamma: float = 0.99
    lam: float = 0.98
    epsilon: float = 0.2
    entropy_beta: float = 0.01
    k_epochs: int = 5
    use_grad_clip: bool = True
    clip_grad: float = 0.5
    matmul_tf32: bool = False   # library GEMMs of the update on TF32 tensor cores (the reference computes in FP32)
    recompute_old_logp: bool = False  # re-evaluate the behaviour log-probabilities with the update's own arithmetic
                                      # before the first epoch (rollouts collected by a lower-precision twin)
    encoder_tf32: bool = False  # every [rows,128] x [128,<=128] product of the update (graph encoders, GAT projections,
                                # policy heads; > 95 % of its FLOPs) forward + backward on the hand-written tcgen05 TF32
                                # kernels instead of library FP32 GEMMs under autograd
    bn_group_envs: int | None = None  # BatchNorm statistics per buffered step AND per group of this many consecutive envs
                                      # (the rollout's Rollout(bn_group_envs=...)): B envs train as B / bn_group_envs
                                      # reference-sized batches side by side; None = per step over all B envs


# grid.y limit of mtfjsp_enc_bn_fwd, the BatchNorm of the update's training path: BatchNorm groups per call
_MAX_BN_GROUPS = 65535


def _obs(bt, name, idx, nxt=False):
    """Observation field of buffered steps `idx`: through the slot table of a RolloutBuffer (each observation stored
    once), or from a plain dict of [T, ...] tensors with separate `*_n` copies (tests replaying reference dumps)."""
    if isinstance(bt, RolloutBuffer):
        return bt.obs(name, idx, nxt)
    return bt[name + "_n" if nxt else name].index_select(0, idx)


def _steps(bt):
    return bt["candidate"].shape[0]


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def allreduce_mean_grads(params, timer=None, weight=None):
    """One flat NCCL/gloo allreduce over every gradient that exists, then the mean.
    timer: optional list that receives a (start, end) CUDA event pair around the collective.
    weight: this rank's share of the mean times the world size (B_local * world / B_total); None = equal shards.  Each
    rank's loss is a mean over ITS envs, so with unequal shards (total_envs % world != 0) the plain mean over ranks would
    over-weight the envs of the smaller shards."""
    ws = _world()
    if ws == 1:
        return 0
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    if weight is not None and weight != 1.0:
        flat.mul_(weight)
    if timer is not None and flat.is_cuda:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        e1.record()
        timer.append((e0, e1))
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat.div_(ws)
    o = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[o:o + n].view_as(g))
        o += n
    return flat.numel() * flat.element_size()


class MAPPOUpdate:
    def __init__(self, job_actor, machine_actor, global_critic, cfg: PPOConfig | None = None, max_rows=1 << 21):
        """max_rows: node rows (steps x envs x N) per forward/backward chunk -- bounds activation memory, see _minibatch."""
        self.job, self.mch, self.critic = job_actor, machine_actor, global_critic
        self.max_rows = max_rows
        self.cfg = cfg or PPOConfig()
        c = self.cfg
        self.job.train_tf32 = self.mch.train_tf32 = self.critic.train_tf32 = bool(c.encoder_tf32)
        mk = lambda net: torch.optim.Adam(net.parameters(), lr=c.lr, eps=c.lr_eps)          # ppo_algorithm.py:57-79
        self.opt_job, self.opt_mch, self.opt_critic = mk(self.job), mk(self.mch), mk(self.critic)
        sch = lambda o: torch.optim.lr_scheduler.StepLR(o, step_size=c.decay_step_size, gamma=c.decay_ratio)
        self.sched = [sch(self.opt_job), sch(self.opt_mch), sch(self.opt_critic)]
        self.allreduce_bytes = 0
        self.allreduce_events = []   # (start, end) CUDA events of every gradient allreduce, for the time-share report
        self._shard_weight = {}      # B_local -> B_local * world / B_total (one tiny allreduce per batch size)

    def _groups_per_step(self, B):
        """BatchNorm groups in one buffered step of B envs."""
        ge = self.cfg.bn_group_envs
        if ge is None:
            return 1
        if ge < 1 or B % ge or B // ge > _MAX_BN_GROUPS:
            raise ValueError("bn_group_envs must divide the env batch into at most %d groups" % _MAX_BN_GROUPS)
        return B // ge

    def _steps_per_chunk(self, steps, B, extra=0):
        """`steps` capped so that (steps + extra) x groups-per-step stays within one BatchNorm call (grouped BatchNorm only:
        with one group per step the chunking is as it always was)."""
        if self.cfg.bn_group_envs is None:
            return steps
        return max(1, min(steps, _MAX_BN_GROUPS // self._groups_per_step(B) - extra))

    def _grad_weight(self, B, device):
        ws = _world()
        if ws == 1:
            return None
        if B not in self._shard_weight:
            tot = torch.tensor([float(B)], dtype=torch.float64, device=device)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
            self._shard_weight[B] = B * ws / float(tot.item())
        return self._shard_weight[B]

    # ---- values and advantages (ppo_algorithm.py:585-703), no gradients ---------------------------------------------
    def _critic_all(self, task_fea, adj_w, adj_src, mf1, mf2):
        """Global critic over all T buffered steps, T BatchNorm groups, chunked by whole steps."""
        T, B, N = task_fea.shape[:3]
        per = self._steps_per_chunk(max(1, (2 * self.max_rows) // (B * N)), B)
        gps = self._groups_per_step(B)
        out = []
        for t0 in range(0, T, per):
            t1 = min(T, t0 + per)
            g = t1 - t0
            v = self.critic.forward(task_fea[t0:t1].reshape(g * B, N, -1), adj_w[t0:t1].reshape(g * B, N, 2),
                                    adj_src[t0:t1].reshape(g * B, N), mf1[t0:t1].reshape(g * B, -1, 6),
                                    mf2[t0:t1].reshape(g * B, -1, 8), groups=g * gps)
            out.append(v.reshape(g, B, 4))
        return torch.cat(out, dim=0)

    def advantages(self, bt):
        c = self.cfg
        with torch.no_grad():
            if isinstance(bt, RolloutBuffer):
                # one critic pass over the observation SLOTS: the value of a step's next state is the value of the slot
                # after its own (same observation, same candidate-machine features, its own BatchNorm group)
                sl = bt.slots
                v_slots = self._critic_all(sl["task_fea"], sl["adj_w"], sl["adj_src"], bt.mach_fea1_of_slots(), sl["mach_fea2"])
                multi_v, multi_v_n = v_slots.index_select(0, bt.slot), v_slots.index_select(0, bt.slot + 1)
            else:
                multi_v = self._critic_all(bt["task_fea"], bt["adj_w"], bt["adj_src"], bt["mach_fea1"], bt["mach_fea2"])
                mf1_n = torch.cat((bt["mach_fea1"][1:], bt["mach_fea1"][-1:]), dim=0)                 # :598-603
                multi_v_n = self._critic_all(bt["task_fea_n"], bt["adj_w_n"], bt["adj_src_n"], mf1_n, bt["mach_fea2_n"])
            jv, mv, jvn, mvn = bt["job_v"], bt["mch_v"], bt["job_v_n"], bt["mch_v_n"]
            # streams in the reference's order mk, pt, tt, it: local values = job[0], mch[0], mch[1], job[1] (:449-451)
            v_loc = torch.stack((jv[..., 0], mv[..., 0], mv[..., 1], jv[..., 1]), dim=-1)
            v_loc_n = torch.stack((jvn[..., 0], mvn[..., 0], mvn[..., 1], jvn[..., 1]), dim=-1)
            adv_loc = gae4(bt["r4"], v_loc, v_loc_n, bt["done"], c.gamma, c.lam)                      # :438-489
            adv_glob = gae4(bt["r4"], multi_v, multi_v_n, bt["done"], c.gamma, c.lam)                 # :491-536
            return dict(adv_loc=adv_loc, adv_glob=adv_glob, tgt_loc=adv_loc + v_loc, tgt_glob=adv_glob + multi_v,
                        multi_v=multi_v, multi_v_n=multi_v_n)

    # ---- one minibatch (ppo_algorithm.py:716-1073) -------------------------------------------------------------------
    def _minibatch(self, bt, adv, idx):
        """One actor step and one critic step on the buffered steps `idx` (in this order).

        Memory: the minibatch is walked in chunks of whole steps (`max_rows` node rows each) with gradient
        accumulation.  Every loss term is a sum over (step, env) divided by S*B, and BatchNorm groups are single
        steps, so the accumulated gradient is the gradient of the unchunked minibatch.  The machine embedding that
        crosses from item i-1 to item i is re-evaluated for the one step a chunk overlaps its predecessor."""
        c = self.cfg
        S = idx.numel()
        B = bt["candidate"].shape[1]
        J, M, H = self.job.J, self.job.M, self.job.H
        N = J * M
        cs = self._steps_per_chunk(max(1, min(S, self.max_rows // (B * N))), B, extra=1)  # the trunk takes one step more
        gps = self._groups_per_step(B)
        take = lambda name, i=idx: bt[name].index_select(0, i)
        mse_sum = lambda a, b: ((a - b) ** 2).sum()
        inv = 1.0 / (S * B)

        def clipped(ratio, a):                                                                      # :800-814
            return torch.min(ratio * a, torch.clamp(ratio, 1 - c.epsilon, 1 + c.epsilon) * a)

        inp = self.job.w["_input"][None, None, :].expand(1, B, H)
        # The reference calls clip_grad_norm_ right after zero_grad and BEFORE backward (:918-930): no gradient
        # exists at that point, so the actors are not clipped.  Reproduced by not clipping them.
        self.opt_job.zero_grad(set_to_none=True)
        self.opt_mch.zero_grad(set_to_none=True)
        dev = bt["candidate"].device
        tot_j = torch.zeros((), device=dev)
        tot_m = torch.zeros((), device=dev)
        chunks = []
        for s0 in range(0, S, cs):
            s1 = min(S, s0 + cs)
            g, ci = s1 - s0, idx[s0:s1]
            # machine trunks first: item i's job head consumes item i-1's machine embedding (:739-768)
            p0 = max(s0 - 1, 0)
            ti = idx[p0:s1]
            nodes_m, pooled_m = self.mch.trunk(take("mach_fea1", ti).reshape(-1, M, 6), _obs(bt, "mach_fea2", ti).reshape(-1, M, 8),
                                               groups=(s1 - p0) * gps)
            pm = pooled_m.reshape(s1 - p0, B, H)
            gm = (torch.cat((inp, pm[:-1]), dim=0) if s0 == 0 else pm[:-1]).reshape(g * B, H)
            if s0 > 0:
                nodes_m, pooled_m = nodes_m[B:], pooled_m[B:]
            tf = _obs(bt, "task_fea", ci).reshape(g * B, N, -1)
            aw, asrc = _obs(bt, "adj_w", ci).reshape(g * B, N, 2), _obs(bt, "adj_src", ci).reshape(g * B, N)
            adst = _enc.ell_invert(asrc)
            chunks.append((ci, tf, aw, asrc, adst))
            prob_j, pooled_o, job_v = self.job.evaluate(tf, aw, asrc, take("candidate", ci).reshape(g * B, J), gm,
                                                        take("job_mask", ci).reshape(g * B, J), groups=g * gps, adj_dst=adst)
            prob_m, mch_v = self.mch.heads(nodes_m, pooled_m, pooled_o, take("mach_mask", ci).reshape(g * B, M))
            prob_j, prob_m = prob_j.reshape(g, B, J), prob_m.reshape(g, B, M)
            job_v, mch_v = job_v.reshape(g, B, 2), mch_v.reshape(g, B, 2)
            dist_j, dist_m = Categorical(probs=prob_j), Categorical(probs=prob_m)                    # :779-783
            ratio_j = torch.exp(dist_j.log_prob(take("a_job", ci).long()) - take("log_a", ci))        # :795
            ratio_m = torch.exp(dist_m.log_prob(take("a_mach", ci).long()) - take("m_log_a", ci))     # :796
            ag, al = adv["adv_glob"].index_select(0, ci), adv["adv_loc"].index_select(0, ci)
            rw = take("rw", ci)
            w_mk, w_ec, w_tt = rw[..., 0], rw[..., 1], rw[..., 2]

            def weighted_global(ratio):                                                             # :820-822, :861-863
                return (w_mk * clipped(ratio, ag[..., 0]) + w_ec * (clipped(ratio, ag[..., 1]) + clipped(ratio, ag[..., 3]))
                        + w_tt * clipped(ratio, ag[..., 2]))

            glob_j, glob_m = weighted_global(ratio_j), weighted_global(ratio_m)
            loc_j = w_mk * clipped(ratio_j, al[..., 0]) + w_ec * clipped(ratio_j, al[..., 3])          # :826-835
            loc_m = w_ec * clipped(ratio_m, al[..., 1]) + w_tt * clipped(ratio_m, al[..., 2])          # :867-876
            tl = adv["tgt_loc"].index_select(0, ci)
            # MSELoss over the whole [S,B] minibatch (:896-907) = sum of squared errors / (S*B)
            crit_j = mse_sum(w_mk * job_v[..., 0], w_mk * tl[..., 0]) + mse_sum(w_ec * job_v[..., 1], w_ec * tl[..., 3])
            crit_m = mse_sum(w_ec * mch_v[..., 0], w_ec * tl[..., 1]) + mse_sum(w_tt * mch_v[..., 1], w_tt * tl[..., 2])
            # job_actor_loss.mean() + machine_actor_loss.mean() (:913-932), this chunk's share
            lj = ((-2 * glob_j - loc_j - c.entropy_beta * dist_j.entropy()).sum() + 0.5 * crit_j) * inv
            lm = ((-2 * glob_m - loc_m - c.entropy_beta * dist_m.entropy()).sum() + 0.5 * crit_m) * inv
            (lj + lm).backward()
            tot_j += lj.detach()
            tot_m += lm.detach()
            del nodes_m, pooled_m, pm, gm, prob_j, prob_m, pooled_o, job_v, mch_v, dist_j, dist_m, ratio_j, ratio_m, glob_j, glob_m, loc_j, loc_m, crit_j, crit_m, lj, lm
        gw = self._grad_weight(B, dev)
        self.allreduce_bytes += allreduce_mean_grads(self.job.parameters() + self.mch.parameters(), self.allreduce_events, gw)
        self.opt_job.step()
        self.opt_mch.step()

        # global critic on the same minibatch (:943-1000): backward, THEN clip, then step
        self.opt_critic.zero_grad(set_to_none=True)
        tot_c = torch.zeros((), device=tot_j.device)
        for ci, tf, aw, asrc, adst in chunks:
            g = ci.numel()
            v_s = self.critic.forward(tf, aw, asrc, take("mach_fea1", ci).reshape(g * B, M, 6),
                                      _obs(bt, "mach_fea2", ci).reshape(g * B, M, 8), groups=g * gps, adj_dst=adst).reshape(g, B, 4)
            tg = adv["tgt_glob"].index_select(0, ci)
            rw = take("rw", ci)
            w_mk, w_ec, w_tt = rw[..., 0], rw[..., 1], rw[..., 2]
            crit = (mse_sum(w_mk * tg[..., 0], w_mk * v_s[..., 0]) + mse_sum(w_ec * tg[..., 1], w_ec * v_s[..., 1])
                    + mse_sum(w_ec * tg[..., 3], w_ec * v_s[..., 3]) + mse_sum(w_tt * tg[..., 2], w_tt * v_s[..., 2])) * inv   # :965-976
            crit.backward()
            tot_c += crit.detach()
            del v_s, crit
        self.allreduce_bytes += allreduce_mean_grads(self.critic.parameters(), self.allreduce_events, gw)
        if c.use_grad_clip:
            torch.nn.utils.clip_grad_norm_(self.critic.parameters(), c.clip_grad)                   # :993-996
        self.opt_critic.step()
        return tot_j, tot_m, tot_c

    def update(self, bt, mini_bs, orders=None, generator=None):
        """bt: dict of [T, B, ...] device tensors (see `collect`).  orders: optional list (one per epoch) of index
        permutations of range(T), for replaying the reference's SubsetRandomSampler draws in tests.
        -> (loss_mean [3], loss_std [3]) over the K epochs: job actor, machine actor, global critic (:1080-1124)."""
        c = self.cfg
        T = _steps(bt)
        dev = bt["candidate"].device
        prev_tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = bool(c.matmul_tf32)
        try:
            if c.recompute_old_logp:
                self.recompute_old_logp(bt)
            return self._update(bt, mini_bs, orders, generator, T, dev)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev_tf32
            # the rollout twins cache re-laid-out copies of some weights (first-layer column blocks, GAT transpose):
            # without this the next rollout would mix stale and fresh weights
            for net in (self.job, self.mch, self.critic):
                if hasattr(net, "refresh_twins"):
                    net.refresh_twins()

    def recompute_old_logp(self, bt):
        """Overwrites bt["log_a"] / bt["m_log_a"] with the log-probabilities of the stored actions under the CURRENT
        weights evaluated by the update's own arithmetic (FP32 library GEMMs, or the tcgen05 training path), in rollout
        order: step t's job head receives the machine embedding of step t-1, the first step of an episode the learned
        `_input` vector (Run.py:316-363).  The reference rolls out and updates with one network, so its importance ratio
        starts at exactly 1; a rollout collected by the TF32 inference twin would otherwise start a few percent off."""
        T, B = bt["candidate"].shape[:2]
        J, M, H = self.job.J, self.job.M, self.job.H
        N = J * M
        cs = self._steps_per_chunk(max(1, self.max_rows // (B * N)), B)
        gps = self._groups_per_step(B)
        ep0 = bt.get("episode_start")
        dev = bt["candidate"].device
        with torch.no_grad():
            inp = self.job.w["_input"].detach()[None, None, :].expand(1, B, H)
            prev = None  # pooled machine embedding of the step before the chunk
            for s0 in range(0, T, cs):
                s1 = min(T, s0 + cs)
                g = s1 - s0
                ii = torch.arange(s0, s1, device=dev)
                nodes_m, pooled_m = self.mch.trunk(bt["mach_fea1"][s0:s1].reshape(-1, M, 6),
                                                   _obs(bt, "mach_fea2", ii).reshape(-1, M, 8), groups=g * gps)
                pm = pooled_m.reshape(g, B, H)
                gm = torch.cat((inp if prev is None else prev, pm[:-1]), dim=0).clone()
                for t in range(s0, s1):
                    first = (t % N == 0) if ep0 is None else bool(ep0[t])
                    if first:
                        gm[t - s0] = inp[0]
                prev = pm[-1:].clone()
                prob_j, pooled_o, _ = self.job.evaluate(
                    _obs(bt, "task_fea", ii).reshape(g * B, N, -1), _obs(bt, "adj_w", ii).reshape(g * B, N, 2),
                    _obs(bt, "adj_src", ii).reshape(g * B, N), bt["candidate"][s0:s1].reshape(g * B, J), gm.reshape(g * B, H),
                    bt["job_mask"][s0:s1].reshape(g * B, J), groups=g * gps)
                prob_m, _ = self.mch.heads(nodes_m, pooled_m, pooled_o, bt["mach_mask"][s0:s1].reshape(g * B, M))
                la = torch.log(prob_j.gather(1, bt["a_job"][s0:s1].reshape(-1, 1).long()).squeeze(-1))
                mla = torch.log(prob_m.gather(1, bt["a_mach"][s0:s1].reshape(-1, 1).long()).squeeze(-1))
                bt["log_a"][s0:s1].copy_(la.reshape(g, B))
                bt["m_log_a"][s0:s1].copy_(mla.reshape(g, B))

    def _update(self, bt, mini_bs, orders, generator, T, dev):
        c = self.cfg
        with nvtx_range("mtfjsp/ppo_advantages"):
            adv = self.advantages(bt)
        per_epoch = []
        for k in range(c.k_epochs):
            if orders is not None:
                perm = torch.as_tensor(orders[k], device=dev, dtype=torch.long)
            elif generator is None:
                perm = torch.randperm(T, device=dev)
            else:
                perm = torch.randperm(T, generator=generator, device=generator.device).to(dev)
            lj, lm, lc = [], [], []
            for s0 in range(0, T, mini_bs):                                                          # BatchSampler(..., drop_last=False)
                with nvtx_range("mtfjsp/ppo_minibatch"):
                    a, b, cc = self._minibatch(bt, adv, perm[s0:s0 + mini_bs])
                lj.append(a); lm.append(b); lc.append(cc)
            per_epoch.append(torch.stack((torch.stack(lj).mean(), torch.stack(lm).mean(), torch.stack(lc).mean())))
        if c.use_lr_decay:
            for s in self.sched:
                s.step()
        pe = torch.stack(per_epoch)
        std = pe.std(dim=0) if c.k_epochs > 1 else torch.full((3,), float("nan"), device=dev)
        return pe.mean(dim=0), std


    def allreduce_ms(self):
        """Device time spent in gradient allreduces since the last call (synchronises)."""
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in self.allreduce_events)
        self.allreduce_events.clear()
        return ms


def collect(rollout, weights_per_episode):
    """Runs len(weights_per_episode) episodes with `rollout` (Run.py:290-545) into a `buffer.RolloutBuffer` (each
    observation stored once; T = episodes * N buffered steps) and returns it: the batch `MAPPOUpdate.update` takes."""
    env = rollout.env
    job, mch = rollout.job, rollout.mch
    if isinstance(job, _enc.EsaJobActor) or isinstance(mch, _enc.EsaMachineActor):
        raise TypeError("the ESA-PPO actors are an evaluation baseline (the reference never trains them): roll them out "
                        "with rollout.Rollout / validate.greedy_validate, not into a PPO buffer")
    buf = RolloutBuffer(len(weights_per_episode), env)
    for w in weights_per_episode:
        collect_episode(rollout, buf, w)
    return buf


def collect_episode(rollout, buf, weights):
    """One episode of `rollout` appended to `buf` (a RolloutBuffer with room for it); weights [B,3] per-env reward weights."""
    env = rollout.env
    job, mch = rollout.job, rollout.mch
    rollout.begin_episode(weights)
    wt = torch.as_tensor(weights, dtype=torch.float32, device=env.device)
    for s in range(env.N):
        buf.store_pre(env, rollout)
        rollout.step()
        buf.store_post(env, rollout, wt)
    t = buf.t
    with torch.no_grad():                                                                            # Run.py:452-475
        _, h_o, jv = job.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, rollout.h_mch, buf["job_mask"][t - 1],
                                  groups=rollout.groups)
        _, _, mv = mch.forward(buf["mach_fea1"][t - 1], env.mach_fea, h_o, buf["mach_mask"][t - 1], groups=rollout.groups)
    buf.store_bootstrap(jv, mv)


def update_from_buffer(rollout, updater, bt, mini_bs=None, generator=None):
    """The PPO update on a filled buffer.  `update` refreshes the rollout's inference twins afterwards, so the next episode
    rolls out with the new weights.  When the rollout runs on a different arithmetic path than the update (TF32 twin vs
    FP32 / tcgen05 training path), the behaviour log-probabilities are re-evaluated on the update's path first
    (MAPPOUpdate.recompute_old_logp).  generator: draws the minibatch orders (MAPPOUpdate.update)."""
    if getattr(rollout.job, "precision", "fp32") != "fp32" and not updater.cfg.recompute_old_logp:
        updater.recompute_old_logp(bt)
    return updater.update(bt, mini_bs or rollout.env.N, generator=generator)


def train_iteration(rollout, updater, weights_per_episode, mini_bs=None):
    """One buffer of experience followed by one PPO update (the body of the reference's training loop, Run.py:530-560)."""
    return update_from_buffer(rollout, updater, collect(rollout, weights_per_episode), mini_bs)
