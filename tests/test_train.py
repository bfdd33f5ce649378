"""End-to-end training (train.Trainer) and the BatchNorm groups of `env_batch` envs it trains with.

CPU: the TrainConfig defaults against the reference's parameters.py, the episode schedule against Run.py's modulo rules,
the top-3 checkpoint bookkeeping, the checkpoint layout against the shipped checkpoints, the MIP CSV reader.
GPU: a grouped rollout against separate reference-sized rollouts (bitwise, eager and CUDA-graph replay), grouped update
gradients against the halves' mean, the groups=B update against the ungrouped one (bitwise), a short training run that
must learn, and checkpoints that reproduce the trainer's last evaluation."""
import importlib
import json
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

GOLD = os.path.join(os.path.dirname(__file__), "golden")
tr = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.train")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")

# parameters.py of the reference (lines 52-60, 74-93, 120-122), pinned here because the tests do not read its tree
REFERENCE_DEFAULTS = dict(n_job=6, n_machine=6, n_edge=2, weights=(0.4, 0.4, 0.2), env_batch=16, resample_freq=5,
                          buffer_size=5, k_epochs=5, eval_freq=10, eval_sample=100, train_seed=0, eval_seed=1, n_train=12800,
                          lr=1e-3, lr_eps=1e-5, use_lr_decay=False, decay_step_size=20, decay_ratio=0.96, gamma=0.99,
                          lam=0.98, entropy_beta=0.01, epsilon=0.2, use_grad_clip=True, clip_grad=0.5, hidden=128)


def test_config_defaults_are_the_references():
    c = tr.TrainConfig()
    for k, v in REFERENCE_DEFAULTS.items():
        assert getattr(c, k) == v, k
    assert c.episodes() == 4000                                    # 12800 / 16 * 5
    p = c.ppo_config()
    assert (p.lr, p.k_epochs, p.bn_group_envs, p.use_lr_decay, p.clip_grad) == (1e-3, 5, 16, False, 0.5)
    assert c.csv_name() == "Obj_100_EvalInstance_J6_M6_E2_BS16_Weight442.csv"


def _reference_schedule(episode_num, resample_freq, buffer_size, eval_freq, N=36):
    """Run.py's loop restated: resample at i % resample_freq == 0 (:190), update when the buffer's step count reaches
    N * buffer_size (:530, the count restarts after each update), evaluate at (i + 1) % eval_freq == 0 or the last (:672)."""
    res, upd, ev = [], [], []
    count = 0
    for i in range(episode_num):
        if i % resample_freq == 0:
            res.append(i)
        for _ in range(N):
            count += 1
            if count == N * buffer_size:
                upd.append(i)
                count = 0
        if (i + 1) % eval_freq == 0 or i == episode_num - 1:
            ev.append(i)
    return res, upd, ev


@pytest.mark.parametrize("E,rf,bs,ef", [(None, 5, 5, 10), (23, 5, 5, 10), (37, 3, 4, 7), (12, 1, 2, 5), (9, 4, 3, 20)])
def test_episode_schedule_follows_run_py(E, rf, bs, ef):
    c = tr.TrainConfig(episode_num=E, resample_freq=rf, buffer_size=bs, eval_freq=ef)
    got = tr.episode_schedule(c)
    assert tuple(got) == _reference_schedule(c.episodes(), rf, bs, ef)
    assert got[2][-1] == c.episodes() - 1                          # the last episode always evaluates
    if E is None:
        assert (len(got[0]), len(got[1]), len(got[2])) == (800, 800, 400)


def test_top3_bookkeeping(tmp_path):
    top = tr.TopCheckpoints()
    objs = [9.0, 7.0, 8.0, 10.0, 3.0, 5.0, 6.0]
    files = {}
    for ep, o in enumerate(objs, start=1):
        names = [str(tmp_path / ("%s_EP%d_.pth" % (p, ep))) for p in ("a", "b")]
        for n in names:
            open(n, "w").write(str(o))
        files[ep] = names
        for n in top.push(o, names):
            os.remove(n)
    left = sorted(os.listdir(tmp_path))
    assert left == sorted(os.path.basename(n) for ep in (5, 6, 7) for n in files[ep])   # objectives 3, 5, 6
    for old, new in top.finish(lambda p, r: p[: p.rindex("_EP")] + "_top%d.pth" % r):
        os.replace(old, new)
    got = {f: open(tmp_path / f).read() for f in os.listdir(tmp_path)}
    assert got == {"a_top1.pth": "3.0", "b_top1.pth": "3.0", "a_top2.pth": "5.0", "b_top2.pth": "5.0",
                   "a_top3.pth": "6.0", "b_top3.pth": "6.0"}


def test_top3_with_fewer_evaluations_names_the_best_top1():
    top = tr.TopCheckpoints()
    top.push(4.0, ["x4"])
    top.push(2.0, ["x2"])
    assert top.finish(lambda p, r: "%s_top%d" % (p, r)) == [("x2", "x2_top1"), ("x4", "x4_top2")]


def test_checkpoints_have_the_shipped_layout(tmp_path):
    """Fresh networks saved as the trainer saves them: key names and shapes of the shipped J6M6E2 checkpoints; they load
    back through validate.load_checkpoint."""
    tab = json.load(open(os.path.join(GOLD, "shipped_checkpoint_keys.json")))
    job = enc.JobActor(tr.init_state_dict(enc.job_actor_keys(128), 0), 6, 6, device="cpu")
    mch = enc.MachineActor(tr.init_state_dict(enc.machine_actor_keys(128), 1), 6, device="cpu")
    crit = enc.GlobalCritic(tr.init_state_dict(enc.global_critic_keys(128), 2), 6, 6, device="cpu")
    for net, f in ((job, "j.pth"), (mch, "m.pth"), (crit, "c.pth")):
        torch.save({k: v.cpu() for k, v in net.state_dict().items()}, tmp_path / f)
    layout = lambda f: {k: list(v.shape) for k, v in torch.load(tmp_path / f, weights_only=True).items()}
    assert layout("j.pth") == tab["PPO_operation_actor_J6M6E2_1000.pth"]
    assert layout("m.pth") == tab["PPO_machine_actor_J6M6E2_1000.pth"]
    assert layout("c.pth") == {k: list(v) for k, v in enc.global_critic_keys(128).items()}
    j2, m2 = val.load_checkpoint(str(tmp_path / "j.pth"), str(tmp_path / "m.pth"), 6, 6, device="cpu")
    for a, b in ((job, j2), (mch, m2)):
        for k, v in a.state_dict().items():
            assert torch.equal(v, b.state_dict()[k]), k


def test_init_state_dict_follows_the_reference_initialisers():
    sd = tr.init_state_dict(enc.machine_actor_keys(128), 4)
    w = sd["m_policy.linears.0.weight"]                            # nn.Linear(384, 128): U(+-1/sqrt(384))
    assert w.abs().max() <= 1 / np.sqrt(384) and w.abs().max() > 0.9 / np.sqrt(384)
    assert torch.equal(sd["bn.weight"], torch.ones(128)) and torch.equal(sd["bn.bias"], torch.zeros(128))
    assert abs(float(sd["gat_layer.W"].std()) - np.sqrt(2 / 256)) < 0.005
    assert torch.equal(sd["gat_layer.W"], tr.init_state_dict(enc.machine_actor_keys(128), 4)["gat_layer.W"])


def test_mip_csv_and_gaps(tmp_path):
    p = tmp_path / "mip.csv"
    p.write_text("runtime,best_objective,Makespan,MachineEC,MachineIdleT,TransEC\n1,2,100,50,10,20\n3,4,200,40,5,25\n")
    mip = val.read_mip_csv(str(p))
    np.testing.assert_array_equal(mip["Makespan"], [100, 200])
    final4 = np.array([[110.0, 55.0, 22.0, 12.0], [200.0, 40.0, 25.0, 5.0]])   # mk, pt, tt, idle
    g, wg = val.mip_gaps(final4, mip)
    np.testing.assert_allclose(g, [[0.1, 0.1, 0.1, 0.2], [0, 0, 0, 0]])
    np.testing.assert_allclose(wg, [0.4 * 0.1 + 0.4 * (0.1 + 0.2) + 0.2 * 0.1, 0.0])


# ---------------------------------------------------------------------------------------------------------------------- GPU
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
ppo = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.ppo")
rules = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rules")


class _JobGrouped(enc.JobActor):
    """The grouped tf32 encoder even at one group (with one group the actor otherwise takes the batch-wide kernels)."""

    def encode(self, task_fea, adj_w, adj_src, groups=1, adj_dst=None):
        return self._encode_tf32_grouped(task_fea.to(torch.float32), adj_w, adj_src, groups)


class _MachGrouped(enc.MachineActor):
    """The grouped tf32 machine trunk even at one group."""

    def trunk(self, machine_fea_1, machine_fea_2, groups=1):
        B, M, H = machine_fea_1.shape[0], self.M, self.H
        a = self.w["gat_layer.a"]
        return self._trunk_tf32_grouped(machine_fea_1.to(torch.float32).reshape(B * M, 6).contiguous(),
                                        machine_fea_2.to(torch.float32).reshape(B * M, 8).contiguous(),
                                        self.w["gat_layer.W"].t().contiguous(), a[0, :H, 0].contiguous(), a[0, H:, 0].contiguous(),
                                        groups)


def _env(d, idx):
    env = envm.BatchedMTFJSPEnv(len(idx), 6, 6, 2, obs_dtype=torch.float32)
    env.load(*(d[k][idx] for k in ("t", "p", "transT", "edge")))
    env.scaler_init()
    return env


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_grouped_rollout_equals_separate_batches(graph):
    """A greedy rollout of B = 16 G envs with bn_group_envs = 16 gives the actions and final costs of G separate 16-env
    rollouts, bit for bit (tf32 actors, the grouped kernels on both sides)."""
    G, E = 3, 16
    B = G * E
    d = ins.synthetic_instances(0, B, 6, 6, 2, 31)
    w = ins.random_weights(0, B, 31)
    sdj, sdm = enc.seeded_state_dict(enc.job_actor_keys(128), 11), enc.seeded_state_dict(enc.machine_actor_keys(128), 12)
    job, mch = _JobGrouped(sdj, 6, 6, precision="tf32"), _MachGrouped(sdm, 6, precision="tf32")

    def run(idx):
        env = _env(d, idx)
        ro = rom.Rollout(env, job, mch, greedy=True, use_cuda_graph=graph, bn_group_envs=E)
        acts = []
        ro.begin_episode(w[idx])
        for _ in range(env.N):
            ro.step()
            acts.append(torch.stack((env.op, env.mach), dim=-1).clone())
        costs = env.costs().clone()
        if graph:                                                  # a second episode of pure replays
            costs2 = ro.run_episode(w[idx]).clone()
            assert torch.equal(costs2, costs)
        return torch.stack(acts).cpu().numpy(), costs.cpu().numpy()

    a_all, c_all = run(np.arange(B))
    for g in range(G):
        a, c = run(np.arange(g * E, (g + 1) * E))
        np.testing.assert_array_equal(a_all[:, g * E:(g + 1) * E], a)
        np.testing.assert_array_equal(c_all[g * E:(g + 1) * E], c)


def _buffer(B, bn_group_envs, seed=5):
    """One FP32 episode of B J6M6 envs with bn_group_envs BatchNorm groups -> the RolloutBuffer."""
    d = ins.synthetic_instances(0, B, 6, 6, 2, seed)
    env = _env(d, np.arange(B))
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 1), 6, 6)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 2), 6)
    ro = rom.Rollout(env, job, mch, greedy=False, seed=3, bn_group_envs=bn_group_envs)
    return ppo.collect(ro, [ins.random_weights(0, B, seed)])


def _plain(bt):
    """The buffer's steps as plain [T, B, ...] tensors (observations of each step included), sliceable by env."""
    plain = {k: v for k, v in bt.items()}
    tt = torch.arange(bt["candidate"].shape[0], device=bt["candidate"].device)
    for name in bt.OBS:
        plain[name] = bt.obs(name, tt)
    return plain


def _nets(bn_group_envs, **kw):
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), 1), 6, 6, trainable=True)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 2), 6, trainable=True)
    crit = enc.GlobalCritic(enc.seeded_state_dict(enc.global_critic_keys(128), 3), 6, 6, trainable=True)
    return ppo.MAPPOUpdate(job, mch, crit, ppo.PPOConfig(bn_group_envs=bn_group_envs, **kw))


def _grads(up):
    """Per network, all its gradients as one vector (zeros where the losses do not reach: the unused fcl_pooling weights).
    Compared as whole vectors: a Linear bias that feeds a BatchNorm has a gradient of zero up to rounding noise."""
    return [torch.cat([(torch.zeros_like(p) if p.grad is None else p.grad).reshape(-1) for p in net.parameters()])
            for net in (up.job, up.mch, up.critic)]


@pytest.mark.gpu
def test_grouped_update_gradients_are_the_mean_of_the_halves():
    """B = 32 with bn_group_envs = 16 against the two 16-env halves, the same advantages and minibatch order, FP32 path:
    one minibatch of every step, learning rate 0 and no clipping so that the gradients are what is compared."""
    rb = _buffer(32, 16)
    up = _nets(16, lr=0.0, use_grad_clip=False)
    with torch.no_grad():
        adv = up.advantages(rb)
    bt = _plain(rb)
    T = bt["candidate"].shape[0]
    idx = torch.randperm(T, generator=torch.Generator().manual_seed(0)).cuda()
    up._minibatch(bt, adv, idx)
    full = _grads(up)
    halves = []
    for s in (slice(0, 16), slice(16, 32)):
        h = _nets(16, lr=0.0, use_grad_clip=False)
        h._minibatch({k: v[:, s] for k, v in bt.items()}, {k: v[:, s] for k, v in adv.items()}, idx)
        halves.append(_grads(h))
    for name, f, a, b in zip(("job actor", "machine actor", "critic"), full, *halves):
        m = (a + b) / 2
        rel = float((f - m).norm()) / float(m.norm())
        assert rel <= 1e-5, (name, rel)


@pytest.mark.gpu
def test_one_group_per_step_equals_the_ungrouped_update():
    """bn_group_envs = B is one BatchNorm group per buffered step, which is what bn_group_envs = None means: the same bits.
    (B = 8: every BatchNorm group fits one block of the statistics kernel, so each run is bitwise repeatable.)"""
    bt = _buffer(8, None, seed=6)
    res = []
    for bge in (None, 8):
        up = _nets(bge, k_epochs=2)
        mean, std = up.update(bt, 12, orders=[np.arange(36)[::-1].copy(), np.arange(36)])
        res.append([p.detach().clone() for p in up.job.parameters() + up.mch.parameters() + up.critic.parameters()] + [mean])
    for a, b in zip(*res):
        assert torch.equal(a, b)


# A short fixed-seed J6M6E2 run: G = 64 reference-sized batches, 120 episodes = 24 updates, evaluations every 20 episodes.
# Two measured runs (NVIDIA B200, 1000 W; before the minibatch order was seeded, so they differ): evaluations
# 775.9 / 734.9 / 710.0 / 711.8 / 700.2 / 703.8 and 724.3 / 713.3 / 716.1 / 716.3 / 699.7 / 696.8, 64-65 s each; FIFO+SPT
# 3006.4 on the same 100 instances; the reference's shipped logs end its 4,000-episode runs at 718-736.  Thresholds:
# a drop of at least 15 from the first evaluation, a last evaluation below 730 and at least 1500 below FIFO+SPT.
LEARN = dict(groups=64, episode_num=120, eval_freq=20, n_train=2048)
LEARN_MIN_DROP = 15.0
LEARN_MAX_LAST = 730.0
LEARN_SLACK_BELOW_FIFO_SPT = 1500.0


@pytest.mark.gpu
def test_short_run_learns_and_checkpoints_reproduce_it(tmp_path):
    cfg = tr.TrainConfig(out_dir=str(tmp_path), **LEARN)
    t = tr.Trainer(cfg, log=print)
    hist = t.run()
    objs = [h["obj_mean"] for h in hist]
    fifo = rules.evaluate_rules(t.eval_set["t"], t.eval_set["p"], t.eval_set["transT"], t.eval_set["edge"], 6, 6, 2,
                                op_rules=("FIFO",), machine_rules=("SPT",))["objective"][0].mean()
    print("eval objective per evaluation %s; FIFO+SPT %.2f; %.1f s" % ([round(o, 2) for o in objs], fifo, t.wall_s))
    assert objs[0] - objs[-1] >= LEARN_MIN_DROP
    assert objs[-1] <= LEARN_MAX_LAST
    assert objs[-1] <= fifo - LEARN_SLACK_BELOW_FIFO_SPT
    files = sorted(os.listdir(tmp_path))
    tag = "J6M6E2"
    for p in tr.NET_FILES:
        for s in ("_final.pth", "_top1.pth", "_top2.pth", "_top3.pth"):
            assert p + tag + s in files
    assert not [f for f in files if "_EP" in f]
    assert len(open(tmp_path / cfg.csv_name()).read().strip().split(",")) == len(hist)
    # the final checkpoint reproduces the last evaluation exactly
    job, mch = val.load_checkpoint(str(tmp_path / ("PPO_job_actor_" + tag + "_final.pth")),
                                   str(tmp_path / ("PPO_machine_actor_" + tag + "_final.pth")), 6, 6)
    r = val.greedy_validate(job, mch, t.eval_set, chunk=cfg.eval_sample)
    np.testing.assert_array_equal(r["final4"], t.last_eval["final4"])
    # the best checkpoint reproduces the best evaluation's objective
    job, mch = val.load_checkpoint(str(tmp_path / ("PPO_job_actor_" + tag + "_top1.pth")),
                                   str(tmp_path / ("PPO_machine_actor_" + tag + "_top1.pth")), 6, 6)
    assert float(val.greedy_validate(job, mch, t.eval_set, chunk=cfg.eval_sample)["objective"].mean()) == min(objs)
