"""Drop-in mirror of the reference's batched environment class.

`Parallel_env` here has the method surface, argument meaning and return layout of
trainer/parallel_env.py:19-282 (the class Run.py:190-665 and algorithm/ppo_algorithm.py:202-317 drive), so the
reference's rollout loop can use it unchanged:

    paral_env = Parallel_env(args)                      # args: the parameters.py dict (SURVEY.md 5.6)
    paral_env.get_batch(dataset_dict)                   # {"t","p","transT","edge"} torch tensors
    paral_env.init_RewardScaling_sameBATCH(shape=4)
    adj, mfea2, tfea = paral_env.init_DGFJSPEnv_state0()
    mfea1 = paral_env.cal_cur_task_machine_feature(task_index, m_mask, tfea)
    adj_, oenv_info, mfea2_, tfea_ = paral_env.DGFJSPEnv_paral_step(joint_actions)
    paral_env.reset_data()

Everything is computed by the sm_100a kernels behind include/mtfjsp.h; this file only moves data and mirrors the
reference's host-side conventions (numpy float64 outputs, python `random` for the per-env reward weights, the
list-of-env objects callers poke into).  `JobMask` mirrors the candidate / job-mask bookkeeping of
algorithm/ppo_algorithm.py:136-188, 202-317, 1126-1165 on top of the kernel-computed masks.
"""
from __future__ import annotations

import random

import numpy as np
import torch

from .env import MASK_ESA, MASK_FINISHED, BatchedMTFJSPEnv


def draw_reward_weights(kind: str, configs: dict):
    """generate_random_weights (singlestep.py:1253-1270): same calls on python's global `random`, same rounding."""
    if kind == "01":
        w = np.array([random.uniform(0, 1) for _ in range(3)])
        return w / np.sum(w, axis=-1)
    if kind == "0.1":
        nums = [round(random.uniform(0, 1), 1) for _ in range(3)]
        total = sum(nums)
        return np.array([round(x / total, 1) for x in nums])
    if kind == "eval":
        return np.array([configs["weight_mk"], configs["weight_ec"], configs["weight_tt"]], dtype=np.float64)
    raise ValueError("Random_weight_type must be '01', '0.1' or 'eval'")


def gantt_text(machine_routes, st, ft, n_machine, width=72):
    """Console Gantt of a schedule: one line per machine with its ops as `task[start,finish)` in route order and a bar
    on a common time axis.  Stands in for the reference's visualizer package (rendering is outside the hot path)."""
    horizon = max([float(ft[int(t) - 1]) for r in machine_routes.values() for t in r] + [1e-9])
    lines = ["makespan %.3f" % (horizon if horizon > 1e-9 else 0.0)]
    for m in range(n_machine):
        route = [int(t) for t in machine_routes.get(m, [])]
        bar = [" "] * width
        for t in route:
            a = int(float(st[t - 1]) / horizon * (width - 1))
            b = max(a + 1, int(float(ft[t - 1]) / horizon * (width - 1)))
            for k in range(a, min(b, width)):
                bar[k] = "#" if bar[k] == " " else "+"
        ops = " ".join("%d[%.1f,%.1f)" % (t, float(st[t - 1]), float(ft[t - 1])) for t in route)
        lines.append("M%-2d |%s| %s" % (m, "".join(bar), ops))
    return "\n".join(lines)


class _ScalerHandle:
    """paral_Rscaling_instance[i]: Run.py:283-284 calls .reset() on each one at the start of an episode."""

    def __init__(self, owner):
        self._owner = owner

    def reset(self):
        self._owner._request_scaler_reset()


class _Nodes:
    def __init__(self, proxy):
        self._p = proxy

    def __getitem__(self, task_id):
        st = self._p._owner._host_state()
        i, b = task_id - 1, self._p._b
        sched = st["mach"][b, i] >= 0
        return {"finish_time": float(st["ft"][b, i]) if sched else None,
                "start_time": float(st["st"][b, i]) if sched else None,
                "machine": int(st["mach"][b, i]),   # -1 while unscheduled, as the reference's node attribute
                "duration": float(self._p._owner.ability_instance[b][0][i][st["mach"][b, i]]) if sched else 0,
                "scheduled": bool(sched), "job": i // self._p._owner.nmachines}


class _Graph:
    def __init__(self, proxy):
        self.nodes = _Nodes(proxy)


class _EnvProxy:
    """paral_env_DG[i]: the attributes the reference's callers read from a single env
    (Run.py:478, 632-633, 653, 660; algorithm/ppo_algorithm.py:271-273)."""

    def __init__(self, owner, b):
        self._owner, self._b = owner, b
        self.G = _Graph(self)

    @property
    def reward_random_weight(self):
        return self._owner._weights[self._b]

    @property
    def makespan_previous_step(self):
        return float(self._owner._host_costs()[self._b, 0])

    @property
    def total_e1_previous_step(self):
        return float(self._owner._host_costs()[self._b, 4])

    @property
    def trans_t_previous_step(self):
        return float(self._owner._host_costs()[self._b, 2])

    @property
    def idle_t_previous_step(self):
        return float(self._owner._host_costs()[self._b, 3])

    @property
    def machine_routes(self):
        r = self._owner._host_state()["routes"][self._b]
        return {m: (r[m][r[m] >= 0] + 1) for m in range(r.shape[0])}

    def reset(self, Random_weight_type="01"):
        # Run.py:660 resets every env after an episode; the observable effect is one more draw of weights
        self._owner._weights[self._b] = draw_reward_weights(Random_weight_type, self._owner.args)
        self._owner._dirty = True

    def render(self, mode="human", *a, **k):
        """Run.py:653: console Gantt of this env's current schedule."""
        st = self._owner._host_state()
        text = gantt_text(self.machine_routes, st["st"][self._b], st["ft"][self._b], self._owner.nmachines)
        if mode == "human":
            print(text)
        return text


class Parallel_env(object):
    def __init__(self, args, device=None, left_shift=True, return_torch=False, compat="dense"):
        """compat="dense" (default): the reference's return types exactly -- `adj` is a dense float64 [B,N,N] array.
        compat="ell": `adj` is the tuple `(adj_w [B,N,2] f32, adj_src [B,N] i16)` of device tensors (compact ELL form,
        10 bytes per op instead of 8 N), the features are device tensors as well and the step info a [B,6] float64 array;
        `compat.ell_to_block_sparse` turns the tuple into the block-diagonal sparse matrix the reference networks build
        from the dense one (INTEGRATION.md has the patch for model/actor_critic.py:134-156).  Nothing but the [B,6] step
        info leaves the device per step."""
        if compat not in ("dense", "ell"):
            raise ValueError("compat must be 'dense' or 'ell'")
        self.compat = compat
        self.njobs = args["n_job"]
        self.nmachines = args["n_machine"]
        self.ntasks = self.njobs * self.nmachines
        self.nedges = args["n_edge"]
        self.batch_size = args["env_batch"]
        self.m_scaling = args.get("m_scaling", 1)
        self.reward_dict = args.get("reward_scaling", {"scaling_divisor": 1})
        self.args = args
        self.ability_instance = []
        self.paral_Rscaling_instance = []
        self.paral_env_DG = []
        self.oenv_info = []
        self.return_torch = return_torch
        self._env = BatchedMTFJSPEnv(
            self.batch_size, self.njobs, self.nmachines, self.nedges, left_shift=left_shift,
            weights=(args.get("weight_mk", 0.4), args.get("weight_ec", 0.4), args.get("weight_tt", 0.2)),
            scaling_divisor=float(self.reward_dict.get("scaling_divisor", 1)), gamma=args.get("GAMMA", 0.99),
            device=device, obs_dtype=torch.float64, mask_mode=MASK_ESA)
        self._weights = np.zeros((self.batch_size, 3))
        self._cache = {}
        self._dirty = True
        self._scaler_reset_pending = False
        self._loaded = False
        self._pin = None

    # ---- reference surface ------------------------------------------------------------------------------------
    def get_batch(self, dataset_dict):
        """trainer/parallel_env.py:39-63.  `edge` may be ragged-free [B,E,W] (pad with -1)."""
        t, p = dataset_dict["t"], dataset_dict["p"]
        tt, edge = dataset_dict["transT"], dataset_dict["edge"]
        as_np = lambda x: x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
        self.ability_instance = [[as_np(t[i]).copy(), as_np(p[i]).copy(), as_np(tt[i]).copy(), as_np(edge[i]).copy()]
                                 for i in range(self.batch_size)]
        self._env.load(t, p, tt, edge)
        self._loaded = True

    def init_RewardScaling_sameBATCH(self, shape):
        assert shape == 4, "the environment emits 4 reward components"
        self._env.scaler_init()
        self.paral_Rscaling_instance = [_ScalerHandle(self) for _ in range(self.batch_size)]

    def init_DGFJSPEnv_state0(self, weights=None, Random_weight_type="01"):
        """trainer/parallel_env.py:87-142: fresh envs, reset (draws the per-env reward weights), initial observation."""
        if not self._loaded:
            raise RuntimeError("get_batch must be called before init_DGFJSPEnv_state0")
        self.paral_env_DG = [_EnvProxy(self, b) for b in range(self.batch_size)]
        if weights is None:
            for b in range(self.batch_size):
                self._weights[b] = draw_reward_weights(Random_weight_type, self.args)
        else:
            self._weights[:] = np.asarray(weights, dtype=np.float64)
        self._env.reset(self._weights)
        self._env.obs(MASK_ESA)
        self._invalidate()
        return self._emit_obs()

    def cal_cur_task_machine_feature(self, task_index, m_mask=None, all_task_fea=None):
        """trainer/parallel_env.py:152-214.  m_mask / all_task_fea are accepted for signature compatibility; the kernel
        reads the same information (infeasible machines, machine of the job predecessor) from the env state."""
        self._flush_scaler_reset()
        op = task_index if torch.is_tensor(task_index) else torch.as_tensor(np.asarray(task_index))
        op = op.to(self._env.device, torch.int32).contiguous()
        m1, _ = self._env.mfea1(op)
        return m1 if self.return_torch else m1.cpu().numpy()

    def DGFJSPEnv_paral_step(self, joint_actions):
        """trainer/parallel_env.py:217-269.  joint_actions: B pairs (task_index, machine_index), 0-based."""
        self._flush_scaler_reset()
        if isinstance(joint_actions, (list, tuple)):  # the reference's list of (task, machine) pairs: twice as fast as asarray
            acts = np.fromiter((v for pair in joint_actions for v in pair), dtype=np.int32, count=2 * self.batch_size)
            acts = acts.reshape(self.batch_size, 2)
        else:
            acts = np.asarray(joint_actions, dtype=np.int32).reshape(self.batch_size, 2)
        dev = self._env.device
        op = torch.as_tensor(np.ascontiguousarray(acts[:, 0])).to(dev)
        mc = torch.as_tensor(np.ascontiguousarray(acts[:, 1])).to(dev)
        self._env.step_obs(op, mc, MASK_ESA)
        self._invalidate()
        if self.compat == "ell":
            e = self._env
            info = torch.cat((e.reward5[:, :1], e.done.to(torch.float64).unsqueeze(1), e.scaled4), dim=1).cpu().numpy()
            e.check_launch_overlap()
            self.oenv_info = info
            if bool(e.invalid.any()):
                print("============= 'DGFJSPEnv_paral_step': invalid (task, machine) for envs",
                      torch.nonzero(e.invalid).flatten().tolist())
            adj, mfea, tfea = self._emit_obs()
            return adj, info, mfea, tfea
        r5 = self._env.reward5.cpu().numpy()
        s4 = self._env.scaled4.cpu().numpy()
        done = self._env.done.cpu().numpy()
        inv = self._env.invalid.cpu().numpy()
        self._env.check_launch_overlap()
        if inv.any():  # the reference prints and corrupts its state; here the step is refused for those envs
            print("============= 'DGFJSPEnv_paral_step': invalid (task, machine) for envs", np.nonzero(inv)[0].tolist())
        rows = np.concatenate([r5[:, :1], done[:, None].astype(np.float64), s4], axis=1).tolist()
        for row, dn in zip(rows, done.tolist()):
            row[1] = bool(dn)
        self.oenv_info = rows
        adj, mfea, tfea = self._emit_obs()
        return adj, self.oenv_info, mfea, tfea

    def reset_data(self):
        self.paral_env_DG = []
        self.oenv_info = []

    # ---- helpers ------------------------------------------------------------------------------------------------
    def _emit_obs(self):
        if self.compat == "ell":   # device tensors, fresh copies (the env rewrites its own buffers in place every step)
            e = self._env
            return ((e.adj_w.clone(), e.adj_src.clone()), e.mach_fea.clone(),
                    e.task_fea.reshape(self.batch_size * self.ntasks, 12).clone())
        adj = self._env.dense_adj(torch.float64)
        tfea = self._env.task_fea.reshape(self.batch_size * self.ntasks, 12)
        mfea = self._env.mach_fea
        if self.return_torch:
            return adj, mfea.clone(), tfea.clone()
        if self._pin is None:  # pinned staging, reused every step: the copies run at PCIe speed
            self._pin = tuple(torch.empty(x.shape, dtype=x.dtype).pin_memory() for x in (adj, mfea, tfea))
        for dst, src in zip(self._pin, (adj, mfea, tfea)):
            dst.copy_(src, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        # fresh arrays, as the reference returns deep copies; torch's CPU copy is multi-threaded, numpy's is not
        return tuple(torch.empty(x.shape, dtype=x.dtype).copy_(x).numpy() for x in self._pin)

    def job_mask_and_candidates(self, mask_mode=MASK_ESA):
        """Kernel-computed equivalent of esa_update_chosenTaskID_CandidateTaskIDx_JobMask's return value."""
        if mask_mode != MASK_ESA:
            self._env.obs(mask_mode)
        cand = self._env.candidate.cpu().numpy().astype(np.int64)
        mask = self._env.job_mask.bool()
        if mask_mode != MASK_ESA:
            mask = mask.clone()
            self._env.obs(MASK_ESA)
        return cand, mask

    def _request_scaler_reset(self):
        self._scaler_reset_pending = True

    def _flush_scaler_reset(self):
        if self._scaler_reset_pending:  # B calls to RewardScaling.reset() collapse into one launch
            self._env.scaler_reset()
            self._scaler_reset_pending = False

    def _invalidate(self):
        self._cache = {}

    def _host_state(self):
        if "state" not in self._cache:
            self._cache["state"] = {k: v.cpu().numpy() for k, v in self._env.export_state().items()}
        return self._cache["state"]

    def _host_costs(self):
        if "costs" not in self._cache:
            c, e1 = self._env.costs(with_total_e1=True)
            self._cache["costs"] = np.concatenate([c.cpu().numpy(), e1.cpu().numpy()[:, None]], axis=1)
        return self._cache["costs"]


class JobMask:
    """Candidate / job-mask bookkeeping with the reference's method names (algorithm/ppo_algorithm.py:202-317,
    1126-1165), answered from the masks the env kernel already computed."""

    def __init__(self, paral_env: Parallel_env, use_esa=True):
        self._pe = paral_env
        self._mode = MASK_ESA if use_esa else MASK_FINISHED
        self.set_to_0()

    def set_to_0(self, *_):
        J, M, B = self._pe.njobs, self._pe.nmachines, self._pe.batch_size
        self.pool_task_dict_batch = [{j: 1 + M * j for j in range(J)} for _ in range(B)]
        self.mask_new_batch = torch.zeros((B, J))

    def initial(self):
        J, M, B = self._pe.njobs, self._pe.nmachines, self._pe.batch_size
        cand = np.tile(np.arange(J) * M, (B, 1))
        return cand, torch.zeros((B, J), dtype=torch.bool, device=self._pe._env.device)

    def esa_update_chosenTaskID_CandidateTaskIDx_JobMask(self, paralenv=None, action_batch=None, mask_value=1):
        return self._pe.job_mask_and_candidates(self._mode)

    Eval_esa_update_chosenTaskID_CandidateTaskIDx_JobMask = esa_update_chosenTaskID_CandidateTaskIDx_JobMask
