"""On-device MAPPO rollout controller (SURVEY.md 8 f-1; reference: Run.py:290-475, algorithm/agent_func.py:22-63).

One rollout step = job actor (GIN encoder + head) -> candidate-machine features -> machine actor (GAT + head) ->
fused env step + observation.  Everything stays on the GPU: sampling is one selection kernel per actor (masked softmax,
counter-based draw, log-probability; `torch.multinomial` above 32 jobs or machines), the
candidate -> op mapping, masks and rewards never visit the host, so there is no host synchronisation inside an
episode (the reference crosses the host/device boundary four times per step).  The whole step can be captured in a
CUDA graph and replayed (`Rollout(..., use_cuda_graph=True)`)."""
from __future__ import annotations

import contextlib
import os

import torch

from .encoder import select as enc_select
from .env import BatchedMTFJSPEnv, MASK_ESA

# MTFJSP_NVTX=1: NVTX ranges around the phases of a rollout step (job encoder + head, candidate-machine features, machine
# actor, env step + observation) for nsys / ncu --nvtx timelines (SURVEY.md 5.1).  Off by default: a range push / pop
# pair costs about a microsecond of host time per phase.
_NVTX = os.environ.get("MTFJSP_NVTX", "0") == "1"


def nvtx_range(name):
    return torch.cuda.nvtx.range(name) if _NVTX else contextlib.nullcontext()


class Rollout:
    def __init__(self, env: BatchedMTFJSPEnv, job_actor, machine_actor, greedy=False, use_cuda_graph=False, seed=0,
                 bn_group_envs=None):
        """bn_group_envs: every BatchNorm of both actors normalises over groups of this many consecutive envs (the
        reference's env_batch), so B = G * bn_group_envs envs roll out as G independent reference-sized batches; None =
        statistics over the whole batch."""
        assert env.obs_dtype == torch.float32, "the actors consume F32 observations"
        self.env, self.job, self.mch = env, job_actor, machine_actor
        if bn_group_envs is not None and (bn_group_envs < 1 or env.B % bn_group_envs):
            raise ValueError("bn_group_envs must divide the env batch")
        self.groups = 1 if bn_group_envs is None else env.B // bn_group_envs
        self.greedy = greedy
        self.gen = torch.Generator(device=env.device)
        self.gen.manual_seed(seed)
        B = env.B
        dev = env.device
        self.h_mch = torch.zeros((B, job_actor.H), dtype=torch.float32, device=dev)
        self.first = True
        # per-step outputs kept for the PPO buffers
        self.log_a = torch.zeros(B, device=dev)
        self.m_log_a = torch.zeros(B, device=dev)
        self.job_v = torch.zeros((B, getattr(job_actor, "n_values", 2)), device=dev)   # 4 for the ESA job actor
        self.mch_v = torch.zeros((B, getattr(machine_actor, "n_values", 2)), device=dev)
        self.use_graph = use_cuda_graph
        self._graph = None
        self._warm = 0
        # sampling by the one-launch selection kernel (encoder.select): counter-based draws keyed by (seed, step counter,
        # env); the counter lives on the device and is advanced inside the step, so CUDA-graph replays draw fresh numbers
        self.fused_select = (not greedy) and env.J <= 32 and env.M <= 32  # one warp lane per job / machine
        self._rng_seed = seed
        self._rng_step = torch.zeros(1, dtype=torch.int64, device=dev)

    def _g(self):
        # graph replays draw from torch's default CUDA generator (capture-aware); eager mode uses the private one
        return None if (self.greedy or self.use_graph) else self.gen

    def begin_episode(self, weights):
        env = self.env
        env.reset(weights)
        env.scaler_reset()
        env.obs(MASK_ESA)
        self.first = True

    def _step_impl(self, first):
        env = self.env
        with torch.no_grad():
            h_in = None if first else self.h_mch
            rng = (self._rng_seed, self._rng_step) if self.fused_select else None
            with nvtx_range("mtfjsp/job_actor"):
                ti, ai, la, prob, h_o, jv = self.job.forward(env.task_fea, env.adj_w, env.adj_src, env.candidate, h_in,
                                                             env.job_mask, greedy=self.greedy, generator=self._g(), rng=rng,
                                                             groups=self.groups)
                env.op.copy_(ti.to(torch.int32))
            with nvtx_range("mtfjsp/mfea1"):
                m1, mmask = env.mfea1(env.op)
            with nvtx_range("mtfjsp/machine_actor"):
                mp, h_m, mv = self.mch.forward(m1, env.mach_fea, h_o, mmask, groups=self.groups, return_logits=rng is not None)
            if rng is not None:
                mp, ma, mla, _ = enc_select(mp, mmask, None, 1.0, False, rng, 1)
                self._rng_step.add_(1)
            elif self.greedy:
                ma = mp.argmax(dim=-1)
            else:
                ma = torch.multinomial(mp, 1, generator=self._g()).squeeze(-1)
            env.mach.copy_(ma.to(torch.int32))
            self.h_mch.copy_(h_m)
            self.log_a.copy_(la)
            self.m_log_a.copy_(mla if rng is not None else torch.log(mp.gather(1, ma.unsqueeze(-1)).squeeze(-1)))
            self.job_v.copy_(jv)
            self.mch_v.copy_(mv)
            with nvtx_range("mtfjsp/env_step_obs"):
                env.step_obs(env.op, env.mach, MASK_ESA)

    def step(self):
        """Advances every env by one operation.  Results: env.reward5 / scaled4 / done / invalid and the new obs."""
        if self.first:
            self._step_impl(True)   # the first step feeds the learnable `_input` instead of a machine embedding
            self.first = False
            return
        if not self.use_graph:
            self._step_impl(False)
            return
        if self._graph is None:
            if self._warm < 1:      # one eager step so every lazy initialisation happens outside the capture
                self._step_impl(False)
                self._warm += 1
                return
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step_impl(False)
            self._graph = g         # capturing records the launches without running them ...
        self._graph.replay()        # ... so the step itself is the replay

    def run_episode(self, weights):
        """Full episode; returns the final costs [B,4] (mk, pt/N, tt, idle) on the device."""
        self.begin_episode(weights)
        for _ in range(self.env.N):
            self.step()
        return self.env.costs()
