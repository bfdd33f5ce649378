"""Import shim + replay driver for the *real* Python reference (read-only, /root/reference).

TEST INFRASTRUCTURE ONLY.  This module exists to (a) validate the C restatement in
``oracle/mtfjsp_oracle.c`` against the reference implementation, (b) generate the golden
vectors committed under ``tests/golden/`` (see ``tests/golden/gen_golden.py``) and (c) time the unmodified
reference (bench.py's cpu_baseline_reference leg).  It reads the reference checkout named by
``$MTFJSP_REFERENCE_ROOT``; the product package never imports it.

Recipe (SURVEY.md Appendix D): three stub packages (gym, matplotlib.pyplot, plotly.figure_factory)
under ``oracle/ref_shims``, a pre-seeded ``graph_jsp_env.wzl_ima_banner`` module, and the reference
roots on ``sys.path``.  ``Parallel_env.get_batch`` is bypassed (it builds a ragged ``np.array`` inside
a log f-string, trainer/parallel_env.py:63) by assigning ``ability_instance`` directly.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("MTFJSP_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "graph-jsp-env", "src", "graph_jsp_env"))


_loaded = {}


def load_reference():
    """Returns a namespace with the reference classes (imported once)."""
    if _loaded:
        return _loaded["ns"]
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    for p in (os.path.join(REF_ROOT, "graph-jsp-env", "src"), REF_ROOT, os.path.join(_HERE, "ref_shims")):
        if p not in sys.path:
            sys.path.insert(0, p)
    banner = types.ModuleType("graph_jsp_env.wzl_ima_banner")
    banner.big_banner = ""
    banner.small_banner = ""
    sys.modules.setdefault("graph_jsp_env.wzl_ima_banner", banner)
    # the reference logs through a module-level logger that prints; keep it quiet
    import io
    import contextlib

    with contextlib.redirect_stdout(io.StringIO()):
        from graph_jsp_env.disjunctive_graph_jsp_env_singlestep import DisjunctiveGraphJspEnv_singleStep
        from trainer.parallel_env import Parallel_env
        from algorithm.ppo_trick import RewardScaling
        from instance.generate_allsize_mofjsp_dataset import Instance_Dataset
    ns = types.SimpleNamespace(
        Env=DisjunctiveGraphJspEnv_singleStep,
        Parallel_env=Parallel_env,
        RewardScaling=RewardScaling,
        Instance_Dataset=Instance_Dataset,
    )
    _loaded["ns"] = ns
    return ns


def make_args(n_job, n_machine, n_edge, env_batch, weights=(0.4, 0.4, 0.2), gamma=0.99):
    """The subset of parameters.py keys the hot path consumes (SURVEY.md 5.6)."""
    return {
        "n_job": n_job,
        "n_machine": n_machine,
        "n_edge": n_edge,
        "env_batch": env_batch,
        "m_scaling": 1,
        "reward_scaling": {"scaling_divisor": 1},
        "GAMMA": gamma,
        "gcn_input_dim": 12,
        "weight_mk": weights[0],
        "weight_ec": weights[1],
        "weight_tt": weights[2],
        "n_total_task": n_job * n_machine,
        "mask_value": 1,
    }


class RefJobMask:
    """The reference's candidate / job-mask bookkeeping, driven exactly as
    algorithm/ppo_algorithm.py:136-188 (init), :202-317 (update) and :1126-1165 (set_to_0) do,
    with the torch.cuda tensors replaced by numpy (no arithmetic is involved on that side)."""

    def __init__(self, n_job, n_machine, batch):
        self.J, self.M, self.B = n_job, n_machine, batch
        self.N = n_job * n_machine
        self.set_to_0()

    def set_to_0(self):
        J, M, B = self.J, self.M, self.B
        self.remaining = [{j: M for j in range(J)} for _ in range(B)]
        self.pool = [{j: 1 + M * j for j in range(J)} for _ in range(B)]
        self.mask_new = np.zeros((B, J))

    def initial(self):
        cand = np.array([list(d.values()) for d in self.pool]) - 1
        return cand, self.mask_new.astype(bool)

    def update(self, paralenv, action_batch, mask_value=1):
        J, M, B, N = self.J, self.M, self.B, self.N
        for b in range(B):
            a = int(action_batch[b])
            if self.remaining[b][a] != 0:
                self.remaining[b][a] -= 1
            if self.remaining[b][a] != 0:
                self.pool[b][a] += 1
            for k, v in self.remaining[b].items():
                if v == 0:
                    self.mask_new[b][k] = mask_value
        mask = self.mask_new.astype(bool).copy()
        for b in range(B):
            G = paralenv.paral_env_DG[b].G
            sel = [0] * N
            ftl = [0] * N
            for i in range(N):
                if G.nodes[i + 1]["finish_time"] is not None:
                    sel[i] = 1
                    ftl[i] = G.nodes[i + 1]["finish_time"]
            sel_np = np.array(sel).reshape(J, M)
            ft_np = np.array(ftl).reshape(J, M)
            colsum = np.sum(sel_np, axis=0)
            rowmax = [max(row) for row in ft_np]
            for c in range(M):
                if c != 0:
                    if colsum[c - 1] == J and colsum[c] != J:
                        for i in range(J):
                            if self.mask_new[b][i] == 1:
                                rowmax[i] = float("inf")
                        mn = min(rowmax)
                        tmp = [1] * J
                        for i, v in enumerate(rowmax):
                            if v == mn:
                                tmp[i] = 0
                        mask[b] = np.array(tmp).astype(bool)
                else:
                    if colsum[c] != J:
                        mask[b] = sel_np[:, c].astype(bool)
        cand = np.array([list(d.values()) for d in self.pool]) - 1
        return cand, mask


def load_ppo_algorithm():
    """The reference's ``algorithm.ppo_algorithm`` module, importable on CPU with two module shims
    (trainer.train_device, trainer.fig_kpi; SURVEY.md Appendix D)."""
    if "ppo" in _loaded:
        return _loaded["ppo"]
    load_reference()
    import contextlib
    import io

    import torch

    td = types.ModuleType("trainer.train_device")
    td.device = torch.device("cpu")
    sys.modules.setdefault("trainer.train_device", td)
    if "trainer.fig_kpi" not in sys.modules:
        fk = types.ModuleType("trainer.fig_kpi")
        fk.get_GPU_usage = lambda *a, **k: None
        fk.result_box_plot = lambda *a, **k: None
        sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from algorithm import ppo_algorithm
    _loaded["ppo"] = ppo_algorithm
    return ppo_algorithm


class RealJobMask:
    """The reference's OWN candidate / job-mask method -- ``PPOAlgorithm.esa_update_chosenTaskID_CandidateTaskIDx_JobMask``
    (algorithm/ppo_algorithm.py:202-317) and ``set_to_0`` (:1126-1165) -- called on an instance made with
    ``object.__new__`` (the constructor builds all networks and calls ``.cuda()``).  The method's own ``.cuda()`` calls
    are answered by a no-op ``Tensor.cuda`` while it runs (this container has no GPU).  Same interface as RefJobMask."""

    def __init__(self, n_job, n_machine, batch):
        pa = load_ppo_algorithm()
        self.J, self.M, self.B = n_job, n_machine, batch
        ppo = object.__new__(pa.PPOAlgorithm)
        ppo.n_job, ppo.n_machine, ppo.n_total_task, ppo.batch_size = n_job, n_machine, n_job * n_machine, batch
        ppo.pool_task_list = [1 + n_machine * i for i in range(n_job)]  # ppo_algorithm.py:158
        self.ppo = ppo
        self.set_to_0()

    class _cpu_cuda:
        def __enter__(self):
            import torch

            self._orig = torch.Tensor.cuda
            torch.Tensor.cuda = lambda t, *a, **k: t
        def __exit__(self, *exc):
            import torch

            torch.Tensor.cuda = self._orig

    def set_to_0(self):
        with self._cpu_cuda():
            self.ppo.set_to_0(None)

    @property
    def mask_new(self):
        return self.ppo.mask_new_batch.numpy()

    def initial(self):
        cand = np.array([list(d.values()) for d in self.ppo.pool_task_dict_batch]) - 1
        return cand, self.ppo.mask_new_batch.bool().numpy().copy()

    def update(self, paralenv, action_batch, mask_value=1):
        import torch

        with self._cpu_cuda():
            cand, mask = self.ppo.esa_update_chosenTaskID_CandidateTaskIDx_JobMask(
                paralenv, torch.as_tensor(np.asarray(action_batch)), mask_value)
        return np.asarray(cand), mask.numpy().copy()


def ref_state_dump(env, N, M):
    """Schedule state of one reference env in array form (0-based op indices)."""
    mach = np.array([env.G.nodes[i + 1]["machine"] for i in range(N)], dtype=np.int32)
    sched = np.array([bool(env.G.nodes[i + 1]["scheduled"]) for i in range(N)])
    st = np.array([env.G.nodes[i + 1]["start_time"] if sched[i] else 0.0 for i in range(N)], dtype=np.float64)
    ft = np.array([env.G.nodes[i + 1]["finish_time"] if sched[i] else 0.0 for i in range(N)], dtype=np.float64)
    routes = np.full((M, N), -1, dtype=np.int32)
    for m in range(M):
        r = np.asarray(env.machine_routes[m]).astype(np.int64) - 1
        routes[m, : len(r)] = r
    return mach, sched, st, ft, routes


def replay(n_job, n_machine, n_edge, t, p, tt, edge, weights, actions=None, left_shift=True, rng=None,
           mask_mode=1, cfg_weights=(0.4, 0.4, 0.2), gamma=0.99, episodes=1, dump_state=True,
           machine_policy="random", obs_steps=None):
    """Runs the reference ``Parallel_env`` on the given instance batch and records every output.

    t, p: [B,N,M]; tt: [B,M,M]; edge: list of B ragged lists (E groups of machine ids);
    weights: [episodes,B,3] per-env reward weights injected after reset (the reference draws them
    from python's global ``random``; injecting keeps the run reproducible);
    actions: optional [episodes,N,B,2] (op, machine); if None, uniformly random valid actions
    under the job mask (mask_mode 1 = ESA rule, 0 = finished-only) are drawn from ``rng``;
    machine_policy "random" | "lowest" | "mixed" picks among the feasible machines;
    obs_steps: optional sorted list of step indices -- the bulky per-step dumps (observation arrays, full schedule
    state) are then kept for those steps only (large instances: a J30M20 episode is 600 steps of 600-row arrays);
    actions, candidate-machine features, step info, candidates and masks are always kept for every step.
    Returns a dict of stacked numpy arrays.
    """
    ref = load_reference()
    B, N, M = t.shape
    J = n_job
    args = make_args(n_job, n_machine, n_edge, B, cfg_weights, gamma)
    pe = ref.Parallel_env(args)
    pe.ability_instance = [[t[b].copy(), p[b].copy(), tt[b].copy(), np.array(edge[b])] for b in range(B)]
    pe.init_RewardScaling_sameBATCH(shape=4)
    out = {k: [] for k in ("adj", "tfea", "mfea2", "mfea1", "info", "cand", "mask", "actions", "mach", "st",
                           "ft", "routes", "costs", "adj0", "tfea0", "mfea20")}
    import torch

    for ep in range(episodes):
        import copy as _copy

        # same construction as parallel_env.py:96-134 but with the left-shift switch exposed
        pe.paral_env_DG = []
        adj_l, tf_l, mf_l = [], [], []
        for b in range(B):
            env = ref.Env(jps_instance=np.array([pe.ability_instance[b][0], pe.ability_instance[b][1]]),
                          reward_function_parameters=args["reward_scaling"],
                          default_visualisations=["gantt_console", "graph_console"], reward_function="wrk",
                          ability_tr_mm=pe.ability_instance[b][2], perform_left_shift_if_possible=left_shift,
                          configs=args)
            pe.paral_env_DG.append(_copy.deepcopy(env))
            e = pe.paral_env_DG[-1]
            e.reset()
            e.reward_random_weight = np.array(weights[ep][b], dtype=np.float64)
            # the initial observation must be rebuilt with the injected weights
            _, _, _, adj, _, mfea, tfea, *_ = e._state_array()
            adj_l.append(adj.copy()); tf_l.append(tfea.copy()); mf_l.append(mfea.copy())
        out["adj0"].append(np.array(adj_l)); out["tfea0"].append(np.concatenate(tf_l, 0)); out["mfea20"].append(np.array(mf_l))
        tfea_cur = np.concatenate(tf_l, 0)
        for rs in pe.paral_Rscaling_instance:
            rs.reset()
        # the golden masks / candidates come from the reference's own method; the restated rule (RefJobMask) rides along
        # and must agree with it at every step
        jm = RealJobMask(J, M, B)
        jm_restated = RefJobMask(J, M, B)
        cand, mask = jm.initial()
        c2, m2 = jm_restated.initial()
        assert np.array_equal(cand, c2) and np.array_equal(mask, m2)
        for step in range(N):
            if actions is not None:
                act = np.asarray(actions[ep][step])
                ops = act[:, 0].astype(np.int64); mch = act[:, 1].astype(np.int64)
                jobs = ops // M
            else:
                jobs = np.zeros(B, dtype=np.int64); ops = np.zeros(B, dtype=np.int64); mch = np.zeros(B, dtype=np.int64)
                for b in range(B):
                    if mask_mode == 1:
                        allowed = np.nonzero(~mask[b])[0]
                    else:
                        allowed = np.nonzero(jm.mask_new[b] == 0)[0]
                    jobs[b] = allowed[rng.integers(len(allowed))]
                    ops[b] = cand[b][jobs[b]]
                    feas = np.nonzero(t[b, ops[b]] >= 0)[0]
                    if machine_policy == "lowest" or (machine_policy == "mixed" and rng.random() < 0.5):
                        mch[b] = feas[0]  # forces same-machine chains (coincident / removed job arcs)
                    else:
                        mch[b] = feas[rng.integers(len(feas))]
            mmask = torch.tensor(np.stack([~(t[b, ops[b]] >= 0) for b in range(B)])[:, None, :])
            mfea1 = pe.cal_cur_task_machine_feature(torch.tensor(ops), mmask, tfea_cur)
            adj_, info, mfea2_, tfea_ = pe.DGFJSPEnv_paral_step(list(zip(ops.tolist(), mch.tolist())))
            cand, mask = jm.update(pe, jobs)
            c2, m2 = jm_restated.update(pe, jobs)
            assert np.array_equal(cand, c2) and np.array_equal(mask, m2) and np.array_equal(jm.mask_new, jm_restated.mask_new), \
                ("restated job-mask rule differs from PPOAlgorithm.esa_update_chosenTaskID_CandidateTaskIDx_JobMask", ep, step)
            tfea_cur = tfea_
            out["actions"].append(np.stack([ops, mch], 1)); out["mfea1"].append(mfea1)
            out["info"].append(np.array(info, dtype=np.float64)); out["cand"].append(cand.copy()); out["mask"].append(mask.copy())
            keep = obs_steps is None or step in obs_steps
            if keep:
                out["adj"].append(adj_); out["tfea"].append(tfea_); out["mfea2"].append(mfea2_)
            if dump_state and keep:
                ds = [ref_state_dump(e, N, M) for e in pe.paral_env_DG]
                out["mach"].append(np.stack([d[0] for d in ds])); out["st"].append(np.stack([d[2] for d in ds]))
                out["ft"].append(np.stack([d[3] for d in ds])); out["routes"].append(np.stack([d[4] for d in ds]))
        out["costs"].append(np.array([[e.makespan_previous_step, e.total_e1_previous_step / N,
                                       e.trans_t_previous_step, e.idle_t_previous_step] for e in pe.paral_env_DG]))
    res = {}
    for k, v in out.items():
        if not v:
            continue
        a = np.stack(v)
        if k in ("adj0", "tfea0", "mfea20", "costs"):
            res[k] = a  # [episodes, ...]
        elif obs_steps is not None and k in ("adj", "tfea", "mfea2", "mach", "st", "ft", "routes"):
            res[k] = a.reshape((episodes, len(obs_steps)) + a.shape[1:])
        else:
            res[k] = a.reshape((episodes, N) + a.shape[1:])
    if obs_steps is not None:
        res["obs_steps"] = np.asarray(sorted(obs_steps), dtype=np.int32)
    return res


def default_model_args(n_job, n_machine, n_edge=2, env_batch=1):
    """parameters.py:41-125 defaults that the networks, validate.py and pdrs.py read."""
    a = make_args(n_job, n_machine, n_edge, env_batch)
    a.update({"gcn_layer": 3, "mlp_fea_extract_layer": 3, "gcn_hidden_dim": 128, "learn_eps": False,
              "neighbor_pooling_type": "average", "mlp_actor_layer": 3, "mlp_critic_layer": 3, "critic_input_dim": 128,
              "critic_hidden_dim": 128, "use_orthogonal": False, "machine_hidden_dim": 128, "LAMDA": 0.98, "epsilon": 0.2,
              "ENTROPY_BETA": 0.01, "LR": 1e-3, "lr_eps": 1e-5})
    return a


def shipped_checkpoint_paths(n_job=6, n_machine=6, n_edge=2, episode=1000):
    """tester/IoTJ_MAPPO/PPO_{operation,machine}_actor_J*M*E*_*.pth (the `PPO-G` rows of test_all.py:56-75, 166-167)."""
    base = os.path.join(REF_ROOT, "tester", "IoTJ_MAPPO")
    tag = "J%dM%dE%d_%d.pth" % (n_job, n_machine, n_edge, episode)
    return os.path.join(base, "PPO_operation_actor_" + tag), os.path.join(base, "PPO_machine_actor_" + tag)


def make_reference_ppo(n_job, n_machine, device, op_pth=None, mch_pth=None):
    """A PPOAlgorithm instance holding the REAL actor networks with shipped weights on `device`, built the way
    tests/golden/gen_ppo_golden.py does (object.__new__: the constructor also builds the unrelated ESA networks).
    What trainer/validate.py:60-297 needs from it: job_actor, machine_actor_gcn, Eval_esa_update_..., set_to_0."""
    import contextlib
    import io

    import torch

    load_reference()
    td = types.ModuleType("trainer.train_device")
    td.device = torch.device(device)
    sys.modules["trainer.train_device"] = td
    if "trainer.fig_kpi" not in sys.modules:
        fk = types.ModuleType("trainer.fig_kpi")
        fk.get_GPU_usage = lambda *a, **k: None
        fk.result_box_plot = lambda *a, **k: None
        sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from algorithm import ppo_algorithm
        from model import actor_critic
    args = default_model_args(n_job, n_machine)
    with contextlib.redirect_stdout(io.StringIO()):
        job = actor_critic.Operation_Actor_JointAction_selfCritic(args)
        mch = actor_critic.Machine_Actor_JointAction_selfGAT_selfCritic(args)
    if op_pth is None:
        op_pth, mch_pth = shipped_checkpoint_paths(n_job, n_machine)
    job.load_state_dict(torch.load(op_pth, map_location="cpu"))
    mch.load_state_dict(torch.load(mch_pth, map_location="cpu"))
    ppo = object.__new__(ppo_algorithm.PPOAlgorithm)
    ppo.n_job, ppo.n_machine, ppo.n_total_task, ppo.batch_size = n_job, n_machine, n_job * n_machine, 1
    ppo.pool_task_list = [1 + n_machine * i for i in range(n_job)]
    ppo.job_actor, ppo.machine_actor_gcn = job.to(device), mch.to(device)
    ppo.set_to_0(None)
    return ppo, args
