"""Device-resident rollout buffer with sparse (ELL) adjacency and the 4-stream GAE (SURVEY.md 8 f-2).

The reference's replay buffer keeps two dense float64 adjacencies per buffered step (trainer/replaybuffer.py:31, 36):
29.9 MB each at B = 16 and 122 GB each at B = 65,536 (N = 36, 180 steps).  Here a step stores the env's native
observation ONCE (next-state fields are the following slot): F32 feature rows plus 10 bytes per node of ELL adjacency,
i.e. 2.5 KB per env-step at J6M6 instead of 24.4 KB, and everything stays on the GPU.  `gae4` replaces the python loops of
algorithm/ppo_algorithm.py:438-536; advantage normalisation uses sums that are allreduced across ranks, so sharded
runs normalise over the same [steps, B_total] block a single GPU would (SURVEY.md 8e)."""
from __future__ import annotations


import torch
import torch.distributed as dist

from . import _lib
from ._lib import _ptr, _stream, check


def gae4(r, v, v_next, done, gamma=0.99, lam=0.98, normalize=True):
    """r, v, v_next [T,B,4] f32 (mk, pt, tt, idle), done [T,B] -> advantages [T,B,4] f32.
    With torch.distributed initialised the normalisation statistics are summed over all ranks."""
    T, B, K = r.shape
    assert K == 4
    r, v, v_next = r.contiguous().float(), v.contiguous().float(), v_next.contiguous().float()
    done = done.contiguous().float()
    adv = torch.empty_like(r)
    stats = torch.zeros(8, dtype=torch.float64, device=r.device)
    check(_lib.lib().mtfjsp_gae4(_ptr(r), _ptr(v), _ptr(v_next), _ptr(done), _ptr(adv), _ptr(stats), T, B, gamma, lam,
                                 _stream()), "mtfjsp_gae4")
    if normalize:
        count = float(T * B)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(stats, op=dist.ReduceOp.SUM)
            cnt = torch.tensor([count], dtype=torch.float64, device=r.device)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
            count = float(cnt.item())
        check(_lib.lib().mtfjsp_adv_normalize(_ptr(adv), _ptr(stats), count, T, B, _stream()), "mtfjsp_adv_normalize")
    return adv


class RolloutBuffer(dict):
    """The PPO buffer `ppo.collect` fills and `MAPPOUpdate` reads (reference fields: trainer/replaybuffer.py:18-204).

    Every observation is stored ONCE: an episode of N steps owns N + 1 observation slots (the N pre-step observations
    and the terminal one), so the next-state fields of the reference buffer (`adj_`, `tasks_fea_`, `machine_fea2_`,
    replaybuffer.py:36-52) are the slot after the step's own -- `obs(name, t, nxt=True)` -- instead of a second copy.
    Everything else is one [T, B, ...] tensor per field, reachable as `buf["name"]` (T = episodes * N buffered steps):

        candidate, job_mask, mach_fea1, mach_mask, a_job, a_mach, log_a, m_log_a, job_v, mch_v, job_v_n, mch_v_n,
        r4 (scaled rewards mk, pt, tt, idle), done, rw (per-env reward weights)

    Observation slots (`S = episodes * (N + 1)`): task_fea [S,B,N,12] f32, adj_w [S,B,N,2] f32, adj_src [S,B,N] i16,
    mach_fea2 [S,B,M,8] f32.  2.5 KB per env-step at J6M6 against 2 x 10.4 KB for the reference's dense float64
    adjacencies alone."""

    OBS = ("task_fea", "adj_w", "adj_src", "mach_fea2")

    def __init__(self, episodes, env):
        super().__init__()
        B, N, M, J, dev = env.B, env.N, env.M, env.J, env.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.episodes, self.N, self.B = episodes, N, B
        T, S = episodes * N, episodes * (N + 1)
        self.T, self.t = T, 0
        self.slots = dict(task_fea=torch.empty((S, B, N, 12), **f32), adj_w=torch.empty((S, B, N, 2), **f32),
                          adj_src=torch.empty((S, B, N), dtype=torch.int16, device=dev),
                          mach_fea2=torch.empty((S, B, M, 8), **f32))
        self.update(
            candidate=torch.empty((T, B, J), dtype=torch.int32, device=dev), job_mask=torch.empty((T, B, J), dtype=torch.uint8, device=dev),
            mach_fea1=torch.empty((T, B, M, 6), **f32), mach_mask=torch.empty((T, B, M), dtype=torch.uint8, device=dev),
            a_job=torch.empty((T, B), dtype=torch.int32, device=dev), a_mach=torch.empty((T, B), dtype=torch.int32, device=dev),
            log_a=torch.empty((T, B), **f32), m_log_a=torch.empty((T, B), **f32),
            job_v=torch.empty((T, B, 2), **f32), mch_v=torch.empty((T, B, 2), **f32),
            job_v_n=torch.empty((T, B, 2), **f32), mch_v_n=torch.empty((T, B, 2), **f32),
            r4=torch.empty((T, B, 4), **f32), done=torch.empty((T, B), **f32), rw=torch.empty((T, B, 3), **f32))
        tt = torch.arange(T, device=dev)
        self.slot = tt + torch.div(tt, N, rounding_mode="floor")        # step t of episode e lives in slot e * (N + 1) + s

    # ---- filling (one episode after the other, in step order) -----------------------------------------------------------
    def _store_obs(self, slot, env):
        sl = self.slots
        sl["task_fea"][slot].copy_(env.task_fea); sl["adj_w"][slot].copy_(env.adj_w); sl["adj_src"][slot].copy_(env.adj_src)
        sl["mach_fea2"][slot].copy_(env.mach_fea)

    def store_pre(self, env, rollout=None):
        """BEFORE rollout.step(): the observation, candidates and job mask the actors are about to see."""
        t = self.t
        self._store_obs(t + t // self.N, env)
        self["candidate"][t].copy_(env.candidate); self["job_mask"][t].copy_(env.job_mask)

    def store_post(self, env, rollout, weights):
        """AFTER rollout.step(): actions, log-probs, values, scaled rewards; at an episode's last step also the terminal
        observation.  Run.py:448-451: the value of step s is the next-value of step s - 1."""
        t, N, M = self.t, self.N, env.M
        s = t % N
        self["mach_fea1"][t].copy_(env.mfea1_buf); self["mach_mask"][t].copy_(env.mach_mask)
        self["a_job"][t].copy_(torch.div(env.op, M, rounding_mode="floor")); self["a_mach"][t].copy_(env.mach)
        self["log_a"][t].copy_(rollout.log_a); self["m_log_a"][t].copy_(rollout.m_log_a)
        self["job_v"][t].copy_(rollout.job_v); self["mch_v"][t].copy_(rollout.mch_v)
        if s > 0:
            self["job_v_n"][t - 1].copy_(rollout.job_v); self["mch_v_n"][t - 1].copy_(rollout.mch_v)
        s4 = env.scaled4                                                  # env order mk, idle, pt, tt -> mk, pt, tt, idle
        r4 = self["r4"]
        r4[t, :, 0].copy_(s4[:, 0]); r4[t, :, 1].copy_(s4[:, 2]); r4[t, :, 2].copy_(s4[:, 3]); r4[t, :, 3].copy_(s4[:, 1])
        self["done"][t].copy_(env.done); self["rw"][t].copy_(weights)
        if s == N - 1:
            self._store_obs(t + t // N + 1, env)                          # terminal observation of the episode
        self.t = t + 1

    def store_bootstrap(self, job_v, mch_v):
        """Next-values of the episode's last step from the extra forward on the terminal observation (Run.py:452-475)."""
        self["job_v_n"][self.t - 1].copy_(job_v); self["mch_v_n"][self.t - 1].copy_(mch_v)

    # ---- reading ------------------------------------------------------------------------------------------------------
    def obs(self, name, idx, nxt=False):
        """Observation field `name` of the buffered steps `idx` (LongTensor): their own slots, or the slots after them."""
        return self.slots[name].index_select(0, self.slot.index_select(0, idx) + (1 if nxt else 0))

    def mach_fea1_of_slots(self):
        """Candidate-machine features paired with every observation slot for the global critic: a pre-step slot takes its
        own step's; a terminal slot the NEXT buffered step's (the reference evaluates next-state values with
        `mach_fea1[t + 1]`, the last one with its own, ppo_algorithm.py:598-603)."""
        N, T = self.N, self.T
        S = self.episodes * (N + 1)
        sl = torch.arange(S, device=self.slot.device)
        e, s = torch.div(sl, N + 1, rounding_mode="floor"), sl % (N + 1)
        t = torch.clamp(e * N + s, max=T - 1)                             # terminal slot of episode e -> step (e + 1) * N
        return self["mach_fea1"].index_select(0, t)

    def bytes_per_env_step(self):
        tot = sum(x.element_size() * x[0, 0].numel() for x in self.values())
        obs = sum(x.element_size() * x[0, 0].numel() for x in self.slots.values())
        return tot + obs * (self.N + 1) / self.N

    def advantages(self, gamma=0.99, lam=0.98):
        """Local 4-stream GAE on the stored actor-critic values (ppo_algorithm.py:438-489)."""
        T = self.t
        jv, mv, jvn, mvn = self["job_v"][:T], self["mch_v"][:T], self["job_v_n"][:T], self["mch_v_n"][:T]
        v = torch.stack((jv[..., 0], mv[..., 0], mv[..., 1], jv[..., 1]), dim=-1)
        vn = torch.stack((jvn[..., 0], mvn[..., 0], mvn[..., 1], jvn[..., 1]), dim=-1)
        return gae4(self["r4"][:T], v, vn, self["done"][:T], gamma, lam)
