"""End-to-end MAPPO training on the device: the reference's training run (Run.py:190-815 with the defaults of
parameters.py) as a `Trainer`.

    python -m e2e-mappo-for-mt-fjsp_b200.train --groups 64 --episodes 200 --out-dir runs/j6m6

One episode rolls out B = groups x env_batch envs with the tf32 inference twins of the three networks (rollout.Rollout,
CUDA-graph replay), every BatchNorm normalising over groups of `env_batch` consecutive envs: G reference-sized batches
side by side, each with the statistics the reference's single batch of `env_batch` envs would see.  The PPO update
(ppo.MAPPOUpdate) keeps the same groups.  The schedule is the reference's:

  * every `resample_freq` episodes the next G x env_batch instances of a freshly shuffled training set are loaded
    (the reshuffled DataLoader batch `current_bs_idx`, Run.py:55-60, 199-210) and the reward scalers restart;
  * every episode draws fresh per-env reward weights (singlestep.py:1255-1259);
  * every `buffer_size` episodes one PPO update with mini_bs = N (Run.py:530-560), then the StepLR step when enabled;
  * every `eval_freq` episodes and after the last one a greedy validation of the `eval_sample` instances of `eval_seed`
    with per-instance BatchNorm (Run.py:672-716), the CSV of eval means, `_final` and `_EP{n}_` checkpoints of which only
    the three best stay on disk, renamed `_top1/2/3` at the end (Run.py:733-814).

Under torchrun every rank owns groups / world of the G batches (the update averages gradients across ranks, BatchNorm
statistics stay per group); rank 0 evaluates and writes the files.
"""
from __future__ import annotations

import argparse
import csv
import heapq
import os
import time
from dataclasses import asdict, dataclass, field

import numpy as np
import torch
import torch.distributed as dist

from . import encoder as enc
from . import instances as ins
from .buffer import RolloutBuffer
from .env import BatchedMTFJSPEnv
from .ppo import MAPPOUpdate, PPOConfig, collect_episode, update_from_buffer
from .rollout import Rollout
from .validate import greedy_validate, mip_gaps, read_mip_csv

NET_FILES = ("PPO_job_actor_", "PPO_machine_actor_", "PPO_global_critic_")   # Run.py:134-136


@dataclass
class TrainConfig:
    """Defaults of the reference's parameters.py (the J6M6E2 run it ships results for)."""
    n_job: int = 6
    n_machine: int = 6
    n_edge: int = 2
    weights: tuple = (0.4, 0.4, 0.2)          # weight_mk, weight_ec, weight_tt (evaluation weights)
    env_batch: int = 16
    resample_freq: int = 5
    buffer_size: int = 5
    k_epochs: int = 5
    eval_freq: int = 10
    eval_sample: int = 100
    train_seed: int = 0
    eval_seed: int = 1
    n_train: int = 12800
    episode_num: int | None = None            # None: n_train / env_batch * resample_freq (parameters.py:120-122)
    lr: float = 1e-3
    lr_eps: float = 1e-5
    use_lr_decay: bool = False
    decay_step_size: int = 20
    decay_ratio: float = 0.96
    gamma: float = 0.99
    lam: float = 0.98
    epsilon: float = 0.2
    entropy_beta: float = 0.01
    use_grad_clip: bool = True
    clip_grad: float = 0.5
    hidden: int = 128
    # this project's own settings
    groups: int = 1                           # G reference-sized batches trained side by side: B = G * env_batch envs
    init_seed: int = 0                        # initial weights (PyTorch's default initialisers, seeded)
    rollout_seed: int = 0                     # action draws of the rollout and minibatch orders of the update
    train_instances: str | None = None        # reference instance pickle; None: reference_stream_instances(train_seed)
    eval_instances: str | None = None         # likewise with eval_seed
    mip_csv: str | None = None                # MIP results of the eval instances: gaps are reported when given
    out_dir: str = "."                        # checkpoints and the eval CSV
    use_cuda_graph: bool = True
    eval_precision: str = "fp32"              # arithmetic of the evaluation actors (fp32 = the reference's)
    ppo_extra: dict = field(default_factory=dict)   # further PPOConfig fields (encoder_tf32, matmul_tf32, ...)

    def episodes(self):
        return int(self.n_train / self.env_batch * self.resample_freq) if self.episode_num is None else int(self.episode_num)

    def ppo_config(self):
        return PPOConfig(lr=self.lr, lr_eps=self.lr_eps, use_lr_decay=self.use_lr_decay, decay_step_size=self.decay_step_size,
                         decay_ratio=self.decay_ratio, gamma=self.gamma, lam=self.lam, epsilon=self.epsilon,
                         entropy_beta=self.entropy_beta, k_epochs=self.k_epochs, use_grad_clip=self.use_grad_clip,
                         clip_grad=self.clip_grad, bn_group_envs=self.env_batch, **self.ppo_extra)

    def tag(self):
        return "J%dM%dE%d" % (self.n_job, self.n_machine, self.n_edge)

    def csv_name(self):
        w = "".join(str(int(x * 10)) for x in self.weights)
        return "Obj_100_EvalInstance_J%d_M%d_E%d_BS%d_Weight%s.csv" % (self.n_job, self.n_machine, self.n_edge, self.env_batch, w)


def episode_schedule(cfg: TrainConfig):
    """-> (resample, update, evaluate): sorted episode indices (0-based) at whose start new instances are loaded, and after
    whose rollout an update / an evaluation runs -- the modulo rules of Run.py:190, 530, 672."""
    E = cfg.episodes()
    resample = [e for e in range(E) if e % cfg.resample_freq == 0]
    update = [e for e in range(E) if (e + 1) % cfg.buffer_size == 0]
    evaluate = [e for e in range(E) if (e + 1) % cfg.eval_freq == 0 or e == E - 1]
    return resample, update, evaluate


class TopCheckpoints:
    """The reference's top-3 bookkeeping (Run.py:752-814): a max-heap on the eval objective keeps the three lowest; the
    files of an evaluation that falls out are deleted; `finish` renames the survivors, best first, to _top1, _top2, ...
    (the reference names them from the worst end, which is the same with three survivors)."""

    def __init__(self, keep=3):
        self.keep = keep
        self.heap = []

    def push(self, objective, files):
        """-> the files to delete now."""
        heapq.heappush(self.heap, (-float(objective),) + tuple(files))
        if len(self.heap) > self.keep:
            return list(heapq.heappop(self.heap)[1:])
        return []

    def finish(self, name_of):
        """name_of(file, rank) -> new path; -> [(old, new)] renames, best evaluation first (rank 1)."""
        out = []
        for rank, entry in enumerate(sorted(self.heap, key=lambda e: e[0], reverse=True), start=1):
            out += [(f, name_of(f, rank)) for f in entry[1:]]
        return out


def init_state_dict(keys: dict, seed: int):
    """Fresh weights as the reference's modules initialise them: nn.Linear's default (weight and bias uniform in
    +-1/sqrt(fan_in)), BatchNorm weight 1 / bias 0 and running statistics 0 / 1, the GAT's W and a Xavier-normal
    (gat.py:63-66), `_input` uniform in [-1, 1] (actor_critic.py:70-71).  Seeded numpy draws, so any machine gives the
    same network."""
    rs = np.random.RandomState(seed)
    sd = {}
    for name, shape in keys.items():
        if name.endswith("num_batches_tracked"):
            sd[name] = torch.tensor(0, dtype=torch.int64)
        elif name.endswith("running_var"):
            sd[name] = torch.ones(shape)
        elif name.endswith("running_mean"):
            sd[name] = torch.zeros(shape)
        elif ".batch_norms." in name or name.startswith("bn.") or ".bn." in name:
            sd[name] = torch.ones(shape) if name.endswith("weight") else torch.zeros(shape)
        elif name == "_input":
            sd[name] = torch.tensor(rs.uniform(-1, 1, size=shape), dtype=torch.float32)
        elif name.startswith("gat_layer."):
            fan_in, fan_out = (shape[1], shape[0]) if len(shape) == 2 else (shape[1] * shape[2], shape[0] * shape[2])
            sd[name] = torch.tensor(rs.normal(0, np.sqrt(2.0 / (fan_in + fan_out)), size=shape), dtype=torch.float32)
        else:
            fan_in = shape[1] if name.endswith("weight") else keys[name[: -len("bias")] + "weight"][1]
            b = 1.0 / np.sqrt(fan_in)
            sd[name] = torch.tensor(rs.uniform(-b, b, size=shape), dtype=torch.float32)
    return sd


def _instances(path, count, J, M, E, seed):
    """The first `count` instances of a reference pickle, or the reference generator's stream `seed`."""
    if path is None:
        return ins.reference_stream_instances(count, J, M, E, seed)
    return {k: v[:count] for k, v in ins.load_instances(path).items()}


def _world():
    return (dist.get_world_size(), dist.get_rank()) if dist.is_available() and dist.is_initialized() else (1, 0)


class Trainer:
    def __init__(self, cfg: TrainConfig, log=print):
        self.cfg = c = cfg
        self.world, self.rank = _world()
        if c.groups % self.world:
            raise ValueError("groups (%d) must be a multiple of the number of ranks (%d)" % (c.groups, self.world))
        self.log = log if self.rank == 0 else (lambda *a, **k: None)
        J, M, E, H = c.n_job, c.n_machine, c.n_edge, c.hidden
        self.N = J * M
        self.G = c.groups // self.world                     # this rank's batches
        self.B = self.G * c.env_batch
        self.env0 = self.rank * self.B                      # first of this rank's envs among all G * env_batch
        self.train = _instances(c.train_instances, c.n_train, J, M, E, c.train_seed)
        if len(self.train["t"]) != c.n_train:
            raise ValueError("the training set holds %d instances, n_train is %d" % (len(self.train["t"]), c.n_train))
        self.eval_set = _instances(c.eval_instances, c.eval_sample, J, M, E, c.eval_seed)
        self.mip = read_mip_csv(c.mip_csv) if c.mip_csv else None
        self.job = enc.JobActor(init_state_dict(enc.job_actor_keys(H), c.init_seed), J, M, hidden=H, trainable=True)
        self.mch = enc.MachineActor(init_state_dict(enc.machine_actor_keys(H), c.init_seed + 1), M, hidden=H, trainable=True)
        self.critic = enc.GlobalCritic(init_state_dict(enc.global_critic_keys(H), c.init_seed + 2), J, M, hidden=H, trainable=True)
        self.env = BatchedMTFJSPEnv(self.B, J, M, E, weights=c.weights, obs_dtype=torch.float32)
        self.rollout = Rollout(self.env, self.job.inference_twin("tf32"), self.mch.inference_twin("tf32"), greedy=False,
                               use_cuda_graph=c.use_cuda_graph, seed=c.rollout_seed + self.rank, bn_group_envs=c.env_batch)
        self.eval_job = self.job.inference_twin(c.eval_precision)
        self.eval_mch = self.mch.inference_twin(c.eval_precision)
        self.updater = MAPPOUpdate(self.job, self.mch, self.critic, c.ppo_config())
        self.order_gen = torch.Generator(device=self.env.device)     # minibatch orders of the updates
        self.order_gen.manual_seed(c.rollout_seed)
        self.history = []       # one dict per evaluation
        self.losses = []        # (episode, loss mean [3], loss std [3]) per update
        self.top = TopCheckpoints()

    # ---- data (Run.py:190-215) ---------------------------------------------------------------------------------------
    def batch_indices(self, k):
        """Training-set indices of this rank's envs for the k-th resample: positions [k * GB, (k + 1) * GB) (modulo the
        set) of the k-th seeded permutation, GB = groups * env_batch."""
        c = self.cfg
        perm = np.random.default_rng([c.train_seed, k]).permutation(c.n_train)
        GB = c.groups * c.env_batch
        return perm[(k * GB + self.env0 + np.arange(self.B)) % c.n_train]

    def load_batch(self, k):
        idx = self.batch_indices(k)
        self.env.load(*(self.train[n][idx] for n in ("t", "p", "transT", "edge")))
        self.env.scaler_init()

    def episode_weights(self, episode):
        return ins.random_weights(self.env0, self.B, self.cfg.train_seed, episode)

    # ---- evaluation (Run.py:672-751) -----------------------------------------------------------------------------------
    def evaluate(self, episode):
        c = self.cfg
        r = greedy_validate(self.eval_job, self.eval_mch, self.eval_set, weights=c.weights, per_instance_batchnorm=True,
                            chunk=c.eval_sample)
        obj, f4 = r["objective"], r["final4"]
        rec = dict(episode=episode + 1, obj_mean=float(obj.mean()), obj_std=float(obj.std()),
                   cost_mean=f4.mean(axis=0).tolist(), cost_std=f4.std(axis=0).tolist())
        if self.mip is not None:
            g, wg = mip_gaps(f4, self.mip, c.weights)
            rec.update(gap_mean=g.mean(axis=0).tolist(), weighted_gap_mean=float(wg.mean()))
        self.history.append(rec)
        self.last_eval = r
        return rec

    def _save(self, suffix):
        os.makedirs(self.cfg.out_dir, exist_ok=True)
        paths = []
        for prefix, net in zip(NET_FILES, (self.job, self.mch, self.critic)):
            p = os.path.join(self.cfg.out_dir, prefix + self.cfg.tag() + suffix)
            torch.save({k: v.cpu() for k, v in net.state_dict().items()}, p)
            paths.append(p)
        return paths

    def record(self, episode, last):
        """The eval CSV and the checkpoints after an evaluation (Run.py:733-814)."""
        c = self.cfg
        os.makedirs(c.out_dir, exist_ok=True)
        with open(os.path.join(c.out_dir, c.csv_name()), "w", newline="") as f:
            csv.writer(f).writerows([[h["obj_mean"] for h in self.history]])
        self._save("_final.pth")
        for p in self.top.push(self.history[-1]["obj_mean"], self._save("_EP%d_.pth" % (episode + 1))):
            os.remove(p)
        if last:
            base = lambda p: p[: p.rindex("_EP")]
            for old, new in self.top.finish(lambda p, rank: base(p) + "_top%d.pth" % rank):
                os.replace(old, new)

    # ---- the run (Run.py:190-815) --------------------------------------------------------------------------------------
    def run(self):
        c = self.cfg
        E = c.episodes()
        resample, update, evaluate = (set(s) for s in episode_schedule(c))
        buf = RolloutBuffer(c.buffer_size, self.env)
        t0 = time.perf_counter()
        env_steps = 0
        for ep in range(E):
            if ep in resample:
                self.load_batch(ep // c.resample_freq)
            collect_episode(self.rollout, buf, self.episode_weights(ep))
            env_steps += self.B * self.N * self.world
            if ep in update:
                mean, std = update_from_buffer(self.rollout, self.updater, buf, self.N, self.order_gen)
                self.losses.append((ep + 1, mean.tolist(), std.tolist()))
                buf.t = 0
            if ep in evaluate and self.rank == 0:
                rec = self.evaluate(ep)
                self.record(ep, ep == E - 1)
                self.log("episode %d/%d  eval obj %.2f (std %.2f)  mk %.2f pt %.2f tt %.2f idle %.2f%s  %.1f s"
                         % (ep + 1, E, rec["obj_mean"], rec["obj_std"], *rec["cost_mean"],
                            "  gap %.4f" % rec["weighted_gap_mean"] if "weighted_gap_mean" in rec else "",
                            time.perf_counter() - t0))
        torch.cuda.synchronize()
        self.wall_s = time.perf_counter() - t0
        self.env_steps = env_steps
        return self.history


def main(argv=None):
    c = TrainConfig()
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    for f, v in asdict(c).items():
        if isinstance(v, (dict, tuple)):
            continue
        kind = (lambda s: s.lower() in ("1", "true", "yes")) if isinstance(v, bool) else (int if f == "episode_num" else
                                                                                          type(v) if v is not None else str)
        ap.add_argument("--" + f.replace("_", "-"), dest=f, type=kind, default=v)
    ap.add_argument("--episodes", dest="episode_num", type=int)
    ap.add_argument("--weights", type=float, nargs=3, default=c.weights)
    a = ap.parse_args(argv)
    cfg = TrainConfig(**{k: (tuple(v) if k == "weights" else v) for k, v in vars(a).items()})
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not dist.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    tr = Trainer(cfg)
    tr.run()
    tr.log("%d episodes of %d envs in %.1f s: %.3e env-steps/s including evaluation"
           % (cfg.episodes(), cfg.groups * cfg.env_batch, tr.wall_s, tr.env_steps / tr.wall_s))
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
