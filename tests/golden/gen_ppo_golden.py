"""Golden vectors for the PPO update (SURVEY.md 8 f-3), produced by the REAL reference on CPU:

    algorithm/ppo_algorithm.py  PPOAlgorithm.global_update_JointActions_GAT_selfCritic (+ the two GAE helpers)
    trainer/replaybuffer.py     ReplayBuffer
    model/actor_critic.py       the three networks, hidden = 32, weights from encoder.seeded_state_dict

The buffer is filled the way Run.py:290-545 fills it, teacher-forced along the recorded reference trajectory of
tests/golden/replay_j6m6_ls_esa.npz (2 episodes x 36 steps x 4 envs), so the observations need not be stored again.
Stored: the buffer fields the networks produced (log-probs, values), the SubsetRandomSampler draws, the losses and
the updated parameters of the three networks after K_epochs = 2 x 2 minibatches.

Run in the build container only:  python tests/golden/gen_ppo_golden.py
"""
import contextlib
import importlib
import io
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")

H, K_EPOCHS = 32, 2


def load():
    rh.load_reference()
    td = types.ModuleType("trainer.train_device")
    td.device = torch.device("cpu")
    sys.modules["trainer.train_device"] = td
    fk = types.ModuleType("trainer.fig_kpi")
    fk.get_GPU_usage = lambda *a, **k: None
    fk.result_box_plot = lambda *a, **k: None
    sys.modules["trainer.fig_kpi"] = fk
    with contextlib.redirect_stdout(io.StringIO()):
        from algorithm import ppo_algorithm
        from model import actor_critic
        from model.gcn_mlp import g_pool_cal
        from trainer import replaybuffer
    return ppo_algorithm, actor_critic, g_pool_cal, replaybuffer


def run_update(before_update=None):
    """Fills the reference ReplayBuffer along the recorded trajectory and runs the reference update once.
    before_update(ppo): called with the PPOAlgorithm object right before the update (e.g. to wrap its optimisers).
    -> (out, nets): the arrays of ppo_golden.npz without the updated parameters, and the three reference modules."""
    pa, ac, g_pool_cal, rb = load()
    g = np.load(os.path.join(HERE, "replay_j6m6_ls_esa.npz"))
    J, M = int(g["J"]), int(g["M"])
    N, B, EP = J * M, g["t"].shape[0], g["actions"].shape[0]
    args = {"n_job": J, "n_machine": M, "env_batch": B, "GAMMA": 0.99, "LAMDA": 0.98, "epsilon": 0.2, "ENTROPY_BETA": 0.01,
            "gcn_layer": 3, "mlp_fea_extract_layer": 3, "gcn_input_dim": 12, "gcn_hidden_dim": H, "learn_eps": False,
            "neighbor_pooling_type": "average", "mlp_actor_layer": 3, "mlp_critic_layer": 3, "critic_input_dim": H,
            "critic_hidden_dim": H, "use_orthogonal": False, "machine_hidden_dim": H, "buffer_size": EP,
            "K_epochs": K_EPOCHS, "use_grad_clip": True, "CLIP_GRAD": 0.5, "use_lr_decay": False, "LR": 1e-3, "lr_eps": 1e-5,
            "decay_step_size": 20, "decay_ratio": 0.96}
    with contextlib.redirect_stdout(io.StringIO()):
        job = ac.Operation_Actor_JointAction_selfCritic(args)
        mch = ac.Machine_Actor_JointAction_selfGAT_selfCritic(args)
        crit = ac.Global_Critic_JointAction_GAT(args)
    # pin the critic's state_dict layout (no checkpoint of it is shipped)
    ck = enc.global_critic_keys(H)
    sd = crit.state_dict()
    assert list(sd.keys()) == list(ck.keys()), (list(sd.keys()), list(ck.keys()))
    assert all(tuple(sd[k].shape) == tuple(ck[k]) for k in ck)
    job.load_state_dict(enc.seeded_state_dict(enc.job_actor_keys(H), 11), strict=True)
    mch.load_state_dict(enc.seeded_state_dict(enc.machine_actor_keys(H), 12), strict=True)
    crit.load_state_dict(enc.seeded_state_dict(ck, 13), strict=True)

    ppo = object.__new__(pa.PPOAlgorithm)  # the constructor also builds the unrelated ESA networks and calls .cuda()
    ppo.n_job, ppo.n_machine, ppo.n_total_task, ppo.batch_size = J, M, N, B
    ppo.GAMMA, ppo.LAMDA, ppo.epsilon, ppo.ENTROPY_BETA = args["GAMMA"], args["LAMDA"], args["epsilon"], args["ENTROPY_BETA"]
    ppo.job_actor, ppo.machine_actor_gcn, ppo.global_critic = job, mch, crit
    mk = lambda net: torch.optim.Adam(net.parameters(), lr=args["LR"], eps=args["lr_eps"])   # ppo_algorithm.py:57-79
    ppo.job_actor_optimizer, ppo.machine_actor_optimizer_gcn, ppo.global_critic_optimizer = mk(job), mk(mch), mk(crit)
    sch = lambda o: torch.optim.lr_scheduler.StepLR(o, step_size=args["decay_step_size"], gamma=args["decay_ratio"])
    ppo.job_actor_lr_decay, ppo.machine_actor_lr_decay_gcn, ppo.global_critic_lr_decay = (
        sch(ppo.job_actor_optimizer), sch(ppo.machine_actor_optimizer_gcn), sch(ppo.global_critic_optimizer))
    ppo.global_critic_loss_func = torch.nn.MSELoss()

    gp = g_pool_cal("average", B, N, torch.device("cpu"))
    buf = rb.ReplayBuffer(args)
    t_arr = g["t"]
    job.train(); mch.train(); crit.train()
    for e in range(EP):
        h_m = None
        flag = 0
        for s in range(N):
            if s == 0:
                tfea, adj = g["tfea0"][e], g["adj0"][e].astype(np.float64)
                cand = np.tile(np.arange(J) * M, (B, 1)).astype(np.int64)
                mask = np.zeros((B, J), dtype=bool)
                mfea2 = g["mfea20"][e]
            else:
                tfea, adj = g["tfea"][e, s - 1], g["adj"][e, s - 1].astype(np.float64)
                cand, mask, mfea2 = g["cand"][e, s - 1].astype(np.int64), g["mask"][e, s - 1], g["mfea2"][e, s - 1]
            op, mc = g["actions"][e, s, :, 0].astype(np.int64), g["actions"][e, s, :, 1].astype(np.int64)
            a_job = torch.tensor(op // M)
            mfea1 = g["mfea1"][e, s]
            mmask = torch.tensor(t_arr[np.arange(B), op] < 0).reshape(B, 1, M)                   # Run.py:335-337
            with torch.no_grad():
                _, _, _, prob, h_o, jv = job(tfea, gp, None, adj, cand, h_m, torch.tensor(mask), use_greedy=True)
                mprob, h_m, mv = mch(mfea1, mfea2, h_o, mmask)
            la = torch.log(prob.gather(1, a_job.unsqueeze(-1)).squeeze(-1))
            mla = torch.log(mprob.gather(1, torch.tensor(mc).unsqueeze(-1)).squeeze(-1))
            tfea_, adj_ = g["tfea"][e, s], g["adj"][e, s].astype(np.float64)
            cand_, mask_, mfea2_ = g["cand"][e, s].astype(np.int64), g["mask"][e, s], g["mfea2"][e, s]
            info = g["info"][e, s]
            flag += 1
            if flag > 1:                                                                           # Run.py:448-451
                buf.store_v_next(j_v_=jv, m_v_=mv)
            done = info[:, 1]
            if done.all():                                                                         # Run.py:452-475
                with torch.no_grad():
                    _, _, _, _, h_o_, jv_ = job(tfea_, gp, None, adj_, cand_, h_m, torch.tensor(mask), use_greedy=True)
                    _, _, mv_ = mch(mfea1, mfea2_, h_o_, mmask)
                buf.store_v_next(j_v_=jv_, m_v_=mv_)
                flag = 0
            rw = np.tile(g["weights"][e], (1, 1))
            buf.store_operation(adj, tfea, cand, torch.tensor(mask), a_job, la, info[:, 0], adj_, tfea_, cand_,
                                torch.tensor(mask_), mfea1, mfea2, mfea2_, torch.tensor(mc), mla, None, done, mmask,
                                info[:, 2], info[:, 4], info[:, 5], info[:, 3], rw, jv, mv)
    assert buf.count_operation == EP * N and buf.count_operation_ == EP * N

    draws = []
    base = pa.SubsetRandomSampler

    class Recording(base):
        def __iter__(self):
            idx = list(super().__iter__())
            draws.append(idx)
            return iter(idx)

    pa.SubsetRandomSampler = Recording
    if before_update is not None:
        before_update(ppo)
    torch.manual_seed(2024)
    with contextlib.redirect_stdout(io.StringIO()):
        loss_mean, loss_std = ppo.global_update_JointActions_GAT_selfCritic(buf, EP * N, gp, args, N)
    pa.SubsetRandomSampler = base
    out = {"H": H, "K_epochs": K_EPOCHS, "mini_bs": N, "orders": np.array(draws, dtype=np.int64),
           "loss_mean": np.array(loss_mean, dtype=np.float64), "loss_std": np.array(loss_std, dtype=np.float64),
           "log_a": buf.a_logprob_operation.numpy(), "m_log_a": buf.a_logprob.numpy(),
           "job_v": buf.job_v.numpy(), "mch_v": buf.machine_v.numpy(), "job_v_n": buf.job_v_.numpy(),
           "mch_v_n": buf.machine_v_.numpy(), "mach_mask": buf.mask_machine_.numpy().reshape(EP * N, B, M)}
    return out, (("job", job), ("mch", mch), ("crit", crit))


def main():
    out, nets = run_update()
    for tag, net in nets:
        for k, v in net.state_dict().items():
            if enc._Params.is_parameter(k):
                out["%s/%s" % (tag, k)] = v.detach().numpy().astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "ppo_golden.npz"), **out)
    print("wrote ppo_golden.npz: orders", out["orders"].shape, "loss_mean", out["loss_mean"], "loss_std", out["loss_std"])


if __name__ == "__main__":
    main()
