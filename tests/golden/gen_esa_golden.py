"""Golden data for the ESA-PPO baseline actors (result CSV row 14, `ESA-PPO` greedy).

Reads a checkout of the reference named by MTFJSP_REFERENCE_ROOT, through oracle/ref_harness.py:

    MTFJSP_REFERENCE_ROOT=<checkout> python tests/golden/gen_esa_golden.py            # everything
    MTFJSP_REFERENCE_ROOT=<checkout> python tests/golden/gen_esa_golden.py --no-ref   # keep the stored ref_cpu

Writes esa_golden.npz:
  csv14 [100,4]            row 14 of results/test_results/Real_{MK,PT,TT,IT}_J6_M6_E2_Seed3_Weight442.csv: final
                           (makespan, processing energy / N, transport time, idle time) of the ESA-PPO greedy rollouts the
                           authors ran on their GPU for the 100 shipped test instances
  esa/op/<key>, esa/mch/<key>   tester/ESWA_MPPO/esa_PPO_{operation,machine}_actor_J6M6E2_800.pth (data, not source):
                           the tensors the policy decisions read.  Left out to keep the fixture small: the value
                           heads (`job_critic.*`, `machine_critic.*`; greedy validation discards the values) and
                           `gat_layer.*`, `fcl_pooling.weight` (in the machine actor's state_dict, never read by its
                           forward).  Their shapes are in shipped_esa_checkpoint_keys.json.
  ref_cpu [100,4]          the UNMODIFIED trainer/validate.py esa_validate_cost_gcn_jointActor_GAT with the reference env
                           and the reference ESA networks on the CPU (it and ppo_algorithm.set_to_0 call `.cuda()` on
                           mask tensors; that call is made a no-op here, nothing else is touched)
  H<h>_<case>_<name>       reference esa_Operation_Actor_Critic / esa_Machine_Actor on CPU with `seeded_state_dict`
                           weights, inputs from replay_j6m6_ls_esa.npz; case g1 = one batch of B instances, case gB = B
                           separate batch-1 calls concatenated (what per-instance BatchNorm groups must reproduce)
and shipped_esa_checkpoint_keys.json: key -> shape of all 12 tester/ESWA_MPPO/*.pth files.
"""
import contextlib
import csv
import glob
import io
import json
import os
import random
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from oracle import ref_harness as rh  # noqa: E402
from gen_encoder_golden import configs, load_models  # noqa: E402
import importlib  # noqa: E402

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
ESA_DIR = "tester/ESWA_MPPO"
UNREAD = ("job_critic.", "machine_critic.", "gat_layer.", "fcl_pooling.")  # not stored, see the module docstring


def csv_row(row):
    a = np.zeros((100, 4))
    for k, name in enumerate(("MK", "PT", "TT", "IT")):
        rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "results/test_results/Real_%s_J6_M6_E2_Seed3_Weight442.csv" % name))))
        a[:, k] = [float(x) for x in rows[row][:100]]
    return a


def module_goldens(ac, g_pool_cal, out):
    g = np.load(os.path.join(HERE, "replay_j6m6_ls_esa.npz"))
    J, M = int(g["J"]), int(g["M"])
    N, B = J * M, g["t"].shape[0]
    for H in (128, 32):
        with contextlib.redirect_stdout(io.StringIO()):
            job = ac.esa_Operation_Actor_Critic(configs(J, M, B, H))
            mch = ac.esa_Machine_Actor(configs(J, M, B, H))
        job.load_state_dict(enc.seeded_state_dict(enc.esa_job_actor_keys(H), 21), strict=True)
        mch.load_state_dict(enc.seeded_state_dict(enc.esa_machine_actor_keys(H), 22), strict=True)
        for s in (5, 20):
            tfea, adj = g["tfea"][0, s], g["adj"][0, s].astype(np.float64)
            cand, mask, mfea2 = g["cand"][0, s].astype(np.int64), g["mask"][0, s], g["mfea2"][0, s]
            mfea1 = g["mfea1"][0, s + 1]
            op = g["actions"][0, s + 1][:, 0]
            mmask = torch.tensor(g["t"][np.arange(B), op] < 0)[:, None, :]
            h_m = torch.tensor(np.random.RandomState(s).uniform(-1, 1, size=(B, H)), dtype=torch.float32)
            for case in ("g1", "gB"):
                parts = [slice(0, B)] if case == "g1" else [slice(b, b + 1) for b in range(B)]
                res = []
                for sl in parts:
                    nb = sl.stop - sl.start
                    job.batch_size = nb
                    gp = g_pool_cal("average", nb, N, torch.device("cpu"))
                    with torch.no_grad():
                        _, _, _, prob, hgo, jv = job(tfea.reshape(B, N, -1)[sl].reshape(nb * N, -1), gp, None, adj[sl], cand[sl],
                                                     h_m[sl], torch.tensor(mask[sl]), use_greedy=True)
                        mp, hp, mv = mch(mfea1[sl], mfea2[sl], hgo, mmask[sl])
                        # the pre-mask scores (x10) that `return_logits=True` hands to the selection kernel
                        logits = _machine_logits(mch, mfea1[sl], mfea2[sl], hgo)
                    res.append((prob, hgo, jv, mp, hp, mv, logits))
                k = "H%d_s%02d_%s_" % (H, s, case)
                for i, name in enumerate(("prob", "pooled", "job_v", "mch_prob", "mch_pooled", "mch_v", "mch_logits")):
                    out[k + name] = torch.cat([r[i] for r in res]).numpy()
            k = "H%d_s%02d_" % (H, s)
            out[k + "hgm_in"] = h_m.numpy()
            out[k + "mmask"] = mmask.numpy()[:, 0, :]
            out[k + "step"] = np.array(s)


def _machine_logits(mch, f1, f2, h_pooled_o):
    """esa_Machine_Actor.forward up to `mch_scores * 10` (actor_critic.py:1276-1383), restated with the module's layers."""
    H = mch.machine_hidden_dim
    f1 = torch.as_tensor(f1).float(); f2 = torch.as_tensor(f2).float()
    h1 = mch.bn(mch.m_fea_1_fcl(f1).reshape(-1, H)).reshape(-1, mch.n_machine, H)
    h2 = mch.bn(mch.m_fea_2_fcl(f2).reshape(-1, H)).reshape(-1, mch.n_machine, H)
    hp = (h1.mean(dim=1) + h2.mean(dim=1)) / 2
    x = torch.cat((h1, h2, hp.unsqueeze(1).expand_as(h1), h_pooled_o.unsqueeze(1).expand_as(h1)), dim=-1)
    return mch.m_policy(x).squeeze(-1) * 10


def reference_validation(ac, sd_op, sd_m):
    """final4 [100,4] of the unmodified esa_validate_cost_gcn_jointActor_GAT over the 100 shipped test instances."""
    torch.Tensor.cuda = lambda self, *a, **k: self  # the reference pins a few mask tensors to the GPU with `.cuda()`
    ppo, args = rh.make_reference_ppo(6, 6, "cpu")
    with contextlib.redirect_stdout(io.StringIO()):
        job = ac.esa_Operation_Actor_Critic(args)
        mch = ac.esa_Machine_Actor(args)
        from trainer import validate
    job.load_state_dict(sd_op, strict=True)
    mch.load_state_dict(sd_m, strict=True)
    ppo.esa_job_actor, ppo.esa_machine_actor_gcn = job, mch
    pd = np.load(os.path.join(HERE, "pdr_golden.npz"))
    ds = types.SimpleNamespace(**{k: pd[k] for k in ("t", "p", "transT", "edge")})
    res = []
    for i in range(100):
        random.seed(i)
        with contextlib.redirect_stdout(io.StringIO()):
            _, final4, _ = validate.esa_validate_cost_gcn_jointActor_GAT(ppo, False, ds, i, "random", greedy=True, args=args)
        res.append(final4)
        print("ref_cpu %3d %s" % (i, final4), flush=True)
    return np.array(res, dtype=np.float64)


def main():
    torch.set_num_threads(4)
    ac, g_pool_cal = load_models()
    out = {"csv14": csv_row(14)}
    sd = {}
    for part, name in (("op", "operation"), ("mch", "machine")):
        sd[part] = torch.load(os.path.join(rh.REF_ROOT, ESA_DIR, "esa_PPO_%s_actor_J6M6E2_800.pth" % name), map_location="cpu")
        for k, v in sd[part].items():
            if not k.startswith(UNREAD):
                out["esa/%s/%s" % (part, k)] = v.numpy()
    module_goldens(ac, g_pool_cal, out)
    path = os.path.join(HERE, "esa_golden.npz")
    if "--no-ref" in sys.argv and os.path.exists(path):
        out["ref_cpu"] = np.load(path)["ref_cpu"]
    elif "--no-ref" not in sys.argv:
        out["ref_cpu"] = reference_validation(ac, sd["op"], sd["mch"])
        print("ref_cpu vs csv14: %d / 100 identical" % int((out["ref_cpu"] == out["csv14"]).all(axis=1).sum()))
    np.savez_compressed(path, **out)
    tab = {}
    for f in sorted(glob.glob(os.path.join(rh.REF_ROOT, ESA_DIR, "*.pth"))):
        tab[os.path.basename(f)] = {k: list(v.shape) for k, v in torch.load(f, map_location="cpu").items()}
    json.dump(tab, open(os.path.join(HERE, "shipped_esa_checkpoint_keys.json"), "w"), indent=0)
    print("wrote %s (%d KB)" % (path, os.path.getsize(path) // 1024))


if __name__ == "__main__":
    main()
