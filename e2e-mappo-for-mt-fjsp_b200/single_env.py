"""Single-environment mirror of the reference's gym class, over the same C ABI (include/mtfjsp.h).

`DisjunctiveGraphJspEnv_singleStep` here answers the constructor keywords, `reset(Random_weight_type)` -> 9-tuple and
`step([task_index, machine_index])` -> 14-tuple of
graph-jsp-env/src/graph_jsp_env/disjunctive_graph_jsp_env_singlestep.py:97-130, 1183-1245, 716-974, plus the attributes
its callers read (`machine_routes`, `G.nodes[task_id]`, `*_previous_step`, `reward_random_weight`, `render`,
`network_as_dataframe`, `valid_action_mask`), so the second group of callers of the boundary -- the validation loop
trainer/validate.py:60-297 and the dispatching-rule rollouts tester/pdrs.py:611-839 -- can switch over by importing this
class instead (tests/test_single_env.py runs both, unmodified, against it).

It is a B = 1 handle of the batched environment: every number comes from the sm_100a kernels, this file only moves
data and rebuilds the reference's host-side containers (numpy arrays, python lists, the node-attribute dicts).  For
throughput use `BatchedMTFJSPEnv` / `Parallel_env`; one env per handle is the reference's calling convention, not a
fast path.
"""
from __future__ import annotations

import numpy as np
import torch

from .env import MASK_ESA, BatchedMTFJSPEnv
from .parallel_env import draw_reward_weights, gantt_text


class _Configs:
    """The reference wraps its config dict in an attribute bag (singlestep.py:27-30, 197)."""

    def __init__(self, d):
        self.__dict__.update(d or {})


class _NodeView:
    """`env.G.nodes[task_id]`: the node attributes of SS:582-593 (task ids are 1-based, 0 = source, N+1 = sink)."""

    def __init__(self, env):
        self._e = env

    def __getitem__(self, task_id):
        e = self._e
        N = e.total_tasks_without_dummies
        if task_id == 0 or task_id == N + 1:  # dummy source / sink (SS:538-560)
            return {"machine": -2, "duration": 0, "scheduled": True, "start_time": 0, "finish_time": 0, "job": -1}
        if not 1 <= task_id <= N:
            raise KeyError(task_id)
        st = e._host_state()
        i = task_id - 1
        sched = st["mach"][i] >= 0
        return {"machine": int(st["mach"][i]),   # -1 while unscheduled
                "duration": float(e.jsp_instance[0][i][st["mach"][i]]) if sched else 0,
                "scheduled": bool(sched), "start_time": float(st["st"][i]) if sched else None,
                "finish_time": float(st["ft"][i]) if sched else None, "job": i // e.n_machines}

    def __len__(self):
        return self._e.total_tasks_without_dummies + 2

    def __iter__(self):
        return iter(range(self._e.total_tasks_without_dummies + 2))

    def __call__(self, data=False):
        return [(i, self[i]) for i in self] if data else list(self)


class _GraphView:
    def __init__(self, env):
        self.nodes = _NodeView(env)


class DisjunctiveGraphJspEnv_singleStep:
    """One MT-FJSP instance on the GPU behind the reference's single-env interface."""

    def __init__(self, jps_instance=None, *, reward_function="nasuta", custom_reward_function=None,
                 reward_function_parameters=None, normalize_observation_space=True, flat_observation_space=True,
                 dtype="float32", action_mode="task", env_transform=None, perform_left_shift_if_possible=True,
                 c_map="rainbow", dummy_task_color="tab:gray", default_visualisations=None, visualizer_kwargs=None,
                 verbose=0, ability_tr_mm=None, ability_p2=None, configs=None, device=None):
        if jps_instance is None or ability_tr_mm is None or configs is None:
            raise ValueError("jps_instance [2,N,M], ability_tr_mm [M,M] and configs are required")
        if reward_function != "wrk":
            raise NotImplementedError("only reward_function='wrk' (the MT-FJSP reward, singlestep.py:1051-1171) is provided")
        if action_mode != "task":
            raise NotImplementedError("action_mode must be 'task'")
        if not (normalize_observation_space and flat_observation_space):
            raise NotImplementedError("the callers of the MT-FJSP path use the default flat, normalised `state` vector")
        self.configs = _Configs(configs)
        self._cfg = dict(configs)
        self.n_jobs, self.n_machines = int(configs["n_job"]), int(configs["n_machine"])  # DGenv_func.py:56 reads them from configs too
        self.total_tasks_without_dummies = self.n_jobs * self.n_machines
        self.jsp_instance = np.asarray(jps_instance, dtype=np.float64)
        if self.jsp_instance.shape != (2, self.total_tasks_without_dummies, self.n_machines):
            raise ValueError("jps_instance must be [2, n_job*n_machine, n_machine]")
        self.instance_transT = np.asarray(ability_tr_mm, dtype=np.float64)
        self.instance_processingEnergy = self.jsp_instance[0] * self.jsp_instance[1]   # SS:355-356
        self.perform_left_shift_if_possible = bool(perform_left_shift_if_possible)
        self.dtype = dtype
        self.verbose = verbose
        self.default_visualisations = default_visualisations
        self.reward_function_parameters = reward_function_parameters or {"scaling_divisor": 1}
        J, M, N = self.n_jobs, self.n_machines, self.total_tasks_without_dummies
        self._env = BatchedMTFJSPEnv(
            1, J, M, 1, left_shift=self.perform_left_shift_if_possible,
            weights=(configs.get("weight_mk", 0.4), configs.get("weight_ec", 0.4), configs.get("weight_tt", 0.2)),
            scaling_divisor=float(self.reward_function_parameters.get("scaling_divisor", 1)), gamma=configs.get("GAMMA", 0.99),
            device=device, obs_dtype=torch.float64, mask_mode=MASK_ESA)
        self._env.load(self.jsp_instance[0][None], self.jsp_instance[1][None], self.instance_transT[None],
                       np.arange(M, dtype=np.int32)[None, None, :])
        self._env.scaler_init()
        self._op = torch.zeros(1, dtype=torch.int32, device=self._env.device)
        self._mc = torch.zeros(1, dtype=torch.int32, device=self._env.device)
        self.G = _GraphView(self)
        self.src_task, self.sink_task = 0, N + 1
        self.reward_random_weight = np.array([configs.get("weight_mk", 0.4), configs.get("weight_ec", 0.4),
                                              configs.get("weight_tt", 0.2)], dtype=np.float64)
        self._clear_episode()
        self._env.reset(self.reward_random_weight[None])   # the constructor ends in load_instance (SS:397-714)
        self._env.obs(MASK_ESA)

    # ---- gym-style surface --------------------------------------------------------------------------------------
    def reset(self, Random_weight_type="01"):
        """SS:1183-1245 -> (state, ft_s, it_s, adj, tasks_fea3, machines_fea, tasks_fea12, est_ft, est_pt)."""
        self._clear_episode()
        self.reward_random_weight = draw_reward_weights(Random_weight_type, self._cfg)
        self._env.reset(np.asarray(self.reward_random_weight, dtype=np.float64)[None])
        self._env.obs(MASK_ESA)
        self._cache = {}
        return self._state_array()

    def step(self, joint_action):
        """SS:716-974 -> (state, reward, done, info, r_t, r_idle, r_pt, r_transT, ft_s, it_s, adj, tasks_fea3,
        machines_fea, tasks_fea12).  An invalid (task, machine) pair leaves the schedule untouched and reports
        `valid_action: False` (the reference corrupts its graph in that case, DESIGN.md 2)."""
        a, m = int(joint_action[0]), int(joint_action[1])
        self._op[0], self._mc[0] = a, m
        len_before = len(self.machine_routes[m]) if 0 <= m < self.n_machines else 0
        self._env.step_obs(self._op, self._mc, MASK_ESA)
        self._cache = {}
        r5 = self._env.reward5.cpu().numpy()[0]
        invalid = bool(self._env.invalid.cpu().numpy()[0])
        done = bool(self._env.done.cpu().numpy()[0])
        self._env.check_launch_overlap()
        info = {"action": a}
        if invalid:
            info.update({"valid_action": False, "node_id": a + 1})
        else:
            self.selected_action.append(a)
            self.selected_action_machine.append(m)
            hs = self._host_state()
            pos = int(np.nonzero(hs["routes"][m] == a)[0][0])
            # SS:1546-1560: a left-shift insertion in front of the route goes through _insert_at_index_0 and carries its label
            method = "_insert_at_index_0" if pos == 0 else "_append_at_the_end" if pos == len_before else "left_shift"
            info.update({"start_time": float(hs["st"][a]), "finish_time": float(hs["ft"][a]), "node_id": a + 1,
                         "valid_action": True, "scheduling_method": method, "left_shift": int(method == "left_shift")})
            # idle_this - idle_prev of the step that placed op a, stored into an int64 array (SS:2118-2121: the list of
            # zeros became np.array([0, ...]) at reset, so the assignment truncates toward zero)
            self._it_s[a] = int(np.trunc(-float(r5[2])))
        info["reward_function"] = "wrk"
        state9 = self._state_array()
        res, ft_s, it_s, adj, tasks_fea3, machines_fea, tasks_fea12, _, _ = state9
        if done:
            info["makespan"] = self.makespan_previous_step
            info["gantt_df"] = self.network_as_dataframe()
        return (res, float(r5[0]), done, info, float(r5[1]), float(r5[2]), float(r5[3]), float(r5[4]), ft_s, it_s, adj,
                tasks_fea3, machines_fea, tasks_fea12)

    def render(self, mode="human", show=None, **kwargs):
        """Console Gantt of the current schedule (the reference draws it with its visualizer package, SS:976-1049)."""
        text = gantt_text(self.machine_routes, self._host_state()["st"], self._host_state()["ft"], self.n_machines)
        if mode == "human":
            print(text)
        return text

    def network_as_dataframe(self):
        """SS:2517-2533."""
        import pandas as pd

        hs = self._host_state()
        return pd.DataFrame([{"Task": "Job %d" % (i // self.n_machines), "Start": float(hs["st"][i]),
                              "Finish": float(hs["ft"][i]), "Resource": "Machine %d" % int(hs["mach"][i])}
                             for i in range(self.total_tasks_without_dummies) if hs["mach"][i] >= 0])

    def valid_action_mask(self, action_mode=None):
        """SS:2535-2576: True where scheduling the task has an effect (unscheduled, job predecessor scheduled)."""
        mach = self._host_state()["mach"]
        M = self.n_machines
        return [bool(mach[i] < 0 and (i % M == 0 or mach[i - 1] >= 0)) for i in range(self.total_tasks_without_dummies)]

    # ---- attributes the callers read ---------------------------------------------------------------------------
    @property
    def machine_routes(self):
        """{machine id: array of task ids (1-based) in processing order} (SS:484)."""
        r = self._host_state()["routes"]
        return {m: (r[m][r[m] >= 0] + 1).astype(np.int64) for m in range(self.n_machines)}

    @property
    def makespan_previous_step(self):
        return float(self._host_costs()[0])

    @property
    def total_e1_previous_step(self):
        return float(self._host_costs()[4])

    @property
    def trans_t_previous_step(self):
        return float(self._host_costs()[2])

    @property
    def idle_t_previous_step(self):
        return float(self._host_costs()[3])

    @property
    def job_mask(self):
        """ESA job mask [J] (True = not selectable) and candidates [J] of the current state (kernel-computed twin of
        algorithm/ppo_algorithm.py:321-417 `Eval_esa_update_...`)."""
        return self._env.job_mask.cpu().numpy()[0].astype(bool), self._env.candidate.cpu().numpy()[0].astype(np.int64)

    # ---- helpers -----------------------------------------------------------------------------------------------------
    def _clear_episode(self):
        self.selected_action = []
        self.selected_action_machine = []
        self._it_s = np.zeros(self.total_tasks_without_dummies, dtype=np.int64)
        self._cache = {}

    def _host_state(self):
        if "state" not in self._cache:
            self._cache["state"] = {k: v.cpu().numpy()[0] for k, v in self._env.export_state().items()}
        return self._cache["state"]

    def _host_costs(self):
        if "costs" not in self._cache:
            c, e1 = self._env.costs(with_total_e1=True)
            self._cache["costs"] = np.concatenate([c.cpu().numpy()[0], e1.cpu().numpy()])
        return self._cache["costs"]

    def _state_array(self):
        """SS:2001-2515."""
        N = self.total_tasks_without_dummies
        env = self._env
        tf12 = env.task_fea.cpu().numpy()[0].copy()                       # [N,12] f64, SS:2246-2277
        machines_fea = env.mach_fea.cpu().numpy()[0].copy()               # [M,8]  f64, SS:2315-2354
        adj_wrk = env.dense_adj(torch.float64).cpu().numpy()[0]           # [N,N]  f64, SS:2019-2073
        raw = env.raw_adj().cpu().numpy()[0]                              # [N,N]  int, SS:2019
        sel = np.zeros(N)
        sel[self.selected_action] = 1
        res = np.column_stack((raw.astype(self.dtype), sel))              # SS:2104-2112
        res = np.ravel(res).astype(self.dtype)                            # SS:2505
        hs = self._host_state()
        ft_s = np.where(hs["mach"] >= 0, hs["ft"], 0.0) if self.selected_action else np.array([0] * N)   # SS:2114-2121
        it_s = np.array(self._it_s)
        sched = tf12[:, 3]
        tasks_fea3 = np.stack((tf12[:, 1], np.where(sched > 0, tf12[:, 2], 0.0), sched), axis=1)          # SS:2204-2217
        return res, ft_s, it_s, adj_wrk, tasks_fea3, machines_fea, tf12, tf12[:, 1].copy(), tf12[:, 2].copy()

    def close(self):
        self._env.close()
