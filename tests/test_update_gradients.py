"""Gradients of the PPO update against the reference and against an FP64 restatement of the three networks.

`test_ppo.py` pins the parameters after four Adam steps, and Adam's step `m / (sqrt(v) + eps)` barely depends on a
gradient's scale, so a kernel that returned 3 x the BatchNorm affine gradients passed it.  Here the gradients themselves
are compared:

1. Reference gradients (`tests/golden/ppo_grad_golden.npz`, gen_ppo_grad_golden.py): the first minibatch of the golden
   update (H = 32, J6M6, 4 envs) with learning rate 0 and no clipping, every parameter's gradient (the critic's before
   `clip_grad_norm_`) against the reference's.  CPU variant with the torch restatements of the kernels of test_ppo.py,
   `gpu` variant with the kernels.  Both must fail when the BatchNorm affine gradients are scaled by 1.01.
2. An FP64 restatement of the three networks and of the PPO loss, written from the reference modules
   (model/gcn_mlp.py, model/gat.py, model/actor_critic.py) and never calling encoder.py's code paths, anchored on the CPU
   against encoder_golden.npz (forward) and ppo_grad_golden.npz (gradients).
3. `gpu`: device VJPs of each network (FP32 path and the tcgen05 TF32 path) and whole `_minibatch` gradients against the
   FP64 restatement at the trainer's shapes and at the size edges.
4. `gpu`: the training kernels at their edges -- BatchNorm with large column means and at the 65,535-group limit,
   aggregation forward / backward on real ELL adjacency up to N = 3,356, the GAT attention backward over a grid-stride
   loop of several rows per warp, the selection kernel at R = 1 and R = 32.

Metric per tensor: rel = |g - g_ref| / |g_ref| (2-norms) and elementwise |g - g_ref| <= a max|g_ref| + r |g_ref|.  A Linear
bias that feeds a BatchNorm has a true gradient of 0 (the normalisation removes any shift), so it is bounded against its
network's gradient norm instead; the unused `fcl_pooling` weights must get no gradient.

Measured values (NVIDIA B200, 1000 W power limit) are recorded beside the bounds they set.  The new `gpu` tests take
about 20 s there.
"""
import importlib
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import test_ppo as tp

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
ppo = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.ppo")

NETS = ("job", "mch", "crit")
KEYS = {"job": enc.job_actor_keys, "mch": enc.machine_actor_keys, "crit": enc.global_critic_keys}
SEEDS = {"job": 11, "mch": 12, "crit": 13}


# ---- comparison -----------------------------------------------------------------------------------------------------
def _zero_grad_bias(k):
    """True gradient 0: Linear biases whose output goes straight into a BatchNorm (gcn_mlp.py:153-154, 248), and the last
    bias of a policy head (one shift of every score, which the softmax removes)."""
    return (k.startswith("encoder.feature_extract.mlps.") and ".linears." in k and k.endswith(".bias")) or \
        k in ("o_policy.linears.2.bias", "m_policy.linears.2.bias")


def compare_grads(got, ref, rel=1e-4, a=1e-4, r=1e-4, zero_tol=1e-4):
    """got / ref: {key: tensor or None} of one network.  -> (failures, stats {key: (rel, cosine)}).
    Tensors with a zero true gradient are bounded by zero_tol x the network's gradient norm (of ref)."""
    fails, stats = [], {}
    norm = math.sqrt(sum(float((v.double() ** 2).sum()) for v in ref.values() if v is not None))
    for k, rv in ref.items():
        gv = got.get(k)
        if k.startswith("fcl_pooling"):
            if gv is not None and float(gv.abs().max()) != 0.0:
                fails.append((k, "unused weight got a gradient"))
            continue
        if rv is None or gv is None:
            if (rv is None) != (gv is None):
                fails.append((k, "gradient present on one side only"))
            continue
        g, rr = gv.detach().double().cpu().reshape(-1), rv.detach().double().cpu().reshape(-1)
        d = (g - rr).norm()
        if _zero_grad_bias(k) or float(rr.abs().max()) == 0.0:
            stats[k] = (float(d) / norm, float("nan"))
            if float(d) > zero_tol * norm:
                fails.append((k, "zero-gradient bias off by %.3g of the network norm" % (float(d) / norm)))
            continue
        rn = float(rr.norm())
        e = float(d) / rn if rn > 0 else float(d)
        cos = float(g @ rr) / (float(g.norm()) * rn) if rn > 0 and float(g.norm()) > 0 else float("nan")
        stats[k] = (e, cos)
        if e > rel:
            fails.append((k, "relative error %.3g" % e))
        elif not bool(((g - rr).abs() <= a * float(rr.abs().max()) + r * rr.abs()).all()):
            fails.append((k, "elementwise bound, worst %.3g of max|ref|" % (float((g - rr).abs().max()) / float(rr.abs().max()))))
    return fails, stats


def _worst(stats):
    vals = [v for k, v in stats.items() if not _zero_grad_bias(k)]
    return max(e for e, _ in vals), min(c for _, c in vals)


# ---- part 1: the first minibatch against the reference's gradients --------------------------------------------------
def _golden_grads(tag, pre_clip=True):
    g = np.load(os.path.join(GOLD, "ppo_grad_golden.npz"))
    H = int(g["H"])
    name = "crit_preclip" if (tag == "crit" and pre_clip) else tag
    out = {}
    for k in KEYS[tag](H):
        if enc._Params.is_parameter(k):
            f = "step0/%s/%s" % (name, k)
            out[k] = torch.tensor(g[f]) if f in g.files else None
    return out


def _net_grads(net):
    return {k: (None if t.grad is None else t.grad.detach().clone()) for k, t in net.w.p.items() if enc._Params.is_parameter(k)}


def _kernel_restatements(monkeypatch):
    monkeypatch.setattr(enc, "bn_forward", tp._t_bn_forward)
    monkeypatch.setattr(enc, "bn_backward", tp._t_bn_backward)
    monkeypatch.setattr(enc, "aggregate", tp._t_aggregate)
    monkeypatch.setattr(enc, "graph_mean", lambda h, *a, **k: h.mean(dim=1))
    monkeypatch.setattr(enc, "ell_invert", lambda s: None)
    monkeypatch.setattr(ppo, "gae4", tp._t_gae4)


def _first_minibatch_device(dev):
    """`_minibatch` on the first minibatch of the golden update, lr 0, no clipping -> ({net: grads}, batch, advantages)."""
    bt, p, (J, M) = tp.build_batch(dev)
    H = int(p["H"])
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(H), 11), J, M, hidden=H, device=dev, trainable=True)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(H), 12), M, hidden=H, device=dev, trainable=True)
    crit = enc.GlobalCritic(enc.seeded_state_dict(enc.global_critic_keys(H), 13), J, M, hidden=H, device=dev, trainable=True)
    up = ppo.MAPPOUpdate(job, mch, crit, ppo.PPOConfig(lr=0.0, use_grad_clip=False))
    adv = up.advantages(bt)
    idx = torch.as_tensor(p["orders"][0][: int(p["mini_bs"])], device=dev, dtype=torch.long)
    up._minibatch(bt, adv, idx)
    return {"job": _net_grads(job), "mch": _net_grads(mch), "crit": _net_grads(crit)}, (bt, adv, idx, J, M, H)


# The critic's graph-encoder gradients with an FP32 neighbourhood mean against the reference's FP64 one (measured 1.43e-3
# on the golden minibatch, see the CPU test); every other tensor is held to 1e-4
CRIT_ENCODER_REL = 2e-3


def _check_against_golden(grads, crit_encoder_rel=None):
    fails = []
    for tag in NETS:
        ref = _golden_grads(tag)
        if tag == "crit" and crit_encoder_rel is not None:
            enc_keys = [k for k in ref if k.startswith("encoder.")]
            f, _ = compare_grads({k: grads[tag][k] for k in enc_keys}, {k: ref[k] for k in enc_keys}, rel=crit_encoder_rel,
                                 a=crit_encoder_rel, r=crit_encoder_rel)
            rest = [k for k in ref if k not in enc_keys]
            f2, _ = compare_grads({k: grads[tag][k] for k in rest}, {k: ref[k] for k in rest})
            f += f2
        else:
            f, _ = compare_grads(grads[tag], ref)
        fails += [(tag,) + x for x in f]
    return fails


def _scaled_bn_backward(monkeypatch, factor):
    inner = enc.bn_backward

    def scaled(*a, **k):
        dx, dg, db = inner(*a, **k)
        return dx, dg * factor, db * factor
    monkeypatch.setattr(enc, "bn_backward", scaled)


def _fp64_mean_aggregate(h, adj_w, adj_src, **k):
    """The neighbourhood mean formed in FP64 and rounded once, as gcn_mlp.py:125-149 does (torch.mm on doubles)."""
    return tp._t_aggregate(h.double(), adj_w.double(), adj_src).float()


def test_first_minibatch_gradients_match_reference_with_torch_kernels(monkeypatch):
    """FP32 restatements of the kernels.  Every tensor within 1e-4 except the critic's graph encoder, which lands at 1.4e-3:
    the update forms the neighbourhood mean in FP32 where the reference forms it in FP64, and the critic's encoder
    gradients (a difference of large per-env terms) amplify that rounding.  With the mean formed in FP64 (next check)
    every tensor of all three networks is back within 1e-4 (worst 5.5e-6), so this is the aggregation's precision and not
    a gradient error."""
    _kernel_restatements(monkeypatch)
    grads, _ = _first_minibatch_device(torch.device("cpu"))
    assert not _check_against_golden(grads, crit_encoder_rel=CRIT_ENCODER_REL)
    monkeypatch.setattr(enc, "aggregate", _fp64_mean_aggregate)
    grads, _ = _first_minibatch_device(torch.device("cpu"))
    assert not _check_against_golden(grads), _check_against_golden(grads)
    _scaled_bn_backward(monkeypatch, 1.01)                       # the comparison is not blind to a gradient's scale
    grads, _ = _first_minibatch_device(torch.device("cpu"))
    fails = _check_against_golden(grads, crit_encoder_rel=CRIT_ENCODER_REL)
    assert any("batch_norms" in k or k.startswith("bn.") for _, k, _ in fails), fails


@pytest.mark.gpu
def test_first_minibatch_gradients_match_reference_on_device(monkeypatch):
    """The kernels: the FP32 aggregation kernel gives the critic's graph encoder the same 1.4e-3 as the CPU variant."""
    grads, _ = _first_minibatch_device(torch.device("cuda", 0))
    fails = _check_against_golden(grads, crit_encoder_rel=CRIT_ENCODER_REL)
    assert not fails, fails
    _scaled_bn_backward(monkeypatch, 1.01)
    grads, _ = _first_minibatch_device(torch.device("cuda", 0))
    fails = _check_against_golden(grads, crit_encoder_rel=CRIT_ENCODER_REL)
    assert any("batch_norms" in k or k.startswith("bn.") for _, k, _ in fails), fails


# ---- part 2: FP64 restatement of the three networks (from the reference modules) -----------------------------------
def ell_to_dense(adj_w, adj_src):
    """[B,N,2] / [B,N] ELL rows -> dense adj[dst, src] float64 with the diagonal set (the reference's layout)."""
    B, N, _ = adj_w.shape
    A = torch.zeros((B, N, N), dtype=torch.float64, device=adj_w.device)
    ar = torch.arange(N, device=adj_w.device)
    A[:, ar, ar] = 1.0
    bj, vj = torch.nonzero(adj_w[:, :, 0] != 0, as_tuple=True)
    A[bj, vj, vj - 1] = adj_w[bj, vj, 0].double()
    bm, vm = torch.nonzero(adj_src >= 0, as_tuple=True)
    A[bm, vm, adj_src[bm, vm].long()] = adj_w[bm, vm, 1].double()
    return A


def f64_params(tag, H, seed=None, sd=None, device="cpu"):
    sd = enc.seeded_state_dict(KEYS[tag](H), SEEDS[tag] if seed is None else seed) if sd is None else sd
    return {k: torch.as_tensor(v).to(device=device, dtype=torch.float64).requires_grad_(True)
            for k, v in sd.items() if enc._Params.is_parameter(k)}


def _bn64(x, w, b, groups):
    """nn.BatchNorm1d in training mode (batch statistics, biased variance, eps 1e-5) per group of rows."""
    xs = x.reshape(groups, -1, x.shape[-1])
    var, mean = torch.var_mean(xs, dim=1, unbiased=False, keepdim=True)
    return ((xs - mean) / torch.sqrt(var + 1e-5) * w + b).reshape(x.shape)


def _linear64(rnd):
    """F.linear, or with rnd (the operand rounding of the tcgen05 path, e.g. to TF32) applied to both GEMM operands."""
    return F.linear if rnd is None else (lambda x, W, b=None: F.linear(rnd(x), rnd(W), b))


def _mlp3_tanh64(w, p, x, rnd=None):                                # MLPActor / MLPCritic, gcn_mlp.py:322-434
    """rnd: see f64_graph_cnn; the tcgen05 path runs the two 128 -> 128 layers on rounded operands, the last in FP32."""
    lin = _linear64(rnd)
    h = torch.tanh(lin(x, w[p + "linears.0.weight"], w[p + "linears.0.bias"]))
    h = torch.tanh(lin(h, w[p + "linears.1.weight"], w[p + "linears.1.bias"]))
    return F.linear(h, w[p + "linears.2.weight"], w[p + "linears.2.bias"])


def f64_graph_cnn(w, task_fea, A, groups, rnd=None, trace=None, feed=None):
    """GraphCNN.forward (gcn_mlp.py:160-197) with next_layer (:109-158): dense neighbourhood mean (bmm, then division by
    the in-degree = non-zeros of the row, :125-149), MLP (:238-249: Linear -> BN -> ReLU twice, then Linear), BN, ReLU;
    then the graph mean (:192).  BatchNorm statistics per group of consecutive envs.
    rnd: None = the reference's arithmetic order.  Otherwise the shadow of the tcgen05 path (encoder._encode_tf32 and its
    grouped form): rnd rounds both operands of every Linear, and the first Linear of the second round forms the product
    first and then the weighted neighbourhood mean of the product rows when N <= 128 (the fused aggregation + layer,
    DESIGN.md section 6), the mean first above 128 nodes.  trace: a list that receives the six pre-BatchNorm Linear outputs.
    feed: six tensors that replace those outputs once traced, so that each layer starts from given values (a device run's
    layer outputs: the restatement then checks one layer at a time)."""
    B, N, _ = task_fea.shape
    deg = (A != 0).sum(-1, keepdim=True).double()
    lin = _linear64(rnd)
    h = task_fea.double()
    for l in (0, 1):
        p = "encoder.feature_extract.mlps.%d." % l
        x = h
        for i in (0, 1, 2):
            W, b = w[p + "linears.%d.weight" % i], w[p + "linears.%d.bias" % i]
            if i > 0:
                x = lin(x, W, b)
            elif rnd is not None and l == 1 and N <= 128:
                x = (torch.bmm(A, lin(x, W).reshape(B, N, -1)) / deg).reshape(B * N, -1) + b
            else:
                x = lin((torch.bmm(A, x) / deg).reshape(B * N, -1), W, b)
            if trace is not None:
                trace.append(x)
            if feed is not None:
                x = feed[3 * l + i].double()
            if i < 2:
                x = F.relu(_bn64(x, w[p + "batch_norms.%d.weight" % i], w[p + "batch_norms.%d.bias" % i], groups))
        x = F.relu(_bn64(x, w["encoder.feature_extract.batch_norms.%d.weight" % l], w["encoder.feature_extract.batch_norms.%d.bias" % l],
                         groups))
        h = x.reshape(B, N, -1)
    return h.mean(dim=1), h


def f64_job_evaluate(w, task_fea, A, candidate, h_g_m_pooled, mask, groups, rnd=None, trace=None, feed=None):
    """Operation_Actor_JointAction_selfCritic.forward (actor_critic.py:180-296) without the draw -> prob, pooled, job_v.
    rnd / trace / feed: see f64_graph_cnn.  With rnd, the policy head's first Linear is split into the column blocks of
    encoder._head_tf32: the candidate rows times the first block, plus (pooled, h_g_m_pooled) times the other two applied
    per env as a bias, each product on rounded operands."""
    pooled, nodes = f64_graph_cnn(w, task_fea, A, groups, rnd, trace, feed)
    J, H = candidate.shape[1], nodes.shape[-1]
    cf = torch.gather(nodes, 1, candidate.long().unsqueeze(-1).expand(-1, J, H))             # :197-207
    gm = w["_input"][None, None, :].expand_as(cf) if h_g_m_pooled is None else h_g_m_pooled.unsqueeze(1).expand_as(cf)  # :230-240
    if rnd is None:
        x = torch.cat((cf, pooled.unsqueeze(1).expand_as(cf), gm), dim=-1)                  # :244-247
        s = _mlp3_tanh64(w, "o_policy.", x)
    else:
        lin, W0, p = _linear64(rnd), w["o_policy.linears.0.weight"], "o_policy."
        env_bias = lin(pooled, W0[:, H:2 * H], w[p + "linears.0.bias"]) + lin(gm[:, 0], W0[:, 2 * H:])
        h = torch.tanh(lin(cf, W0[:, :H]) + env_bias.unsqueeze(1))
        h = torch.tanh(lin(h, w[p + "linears.1.weight"], w[p + "linears.1.bias"]))
        s = F.linear(h, w[p + "linears.2.weight"], w[p + "linears.2.bias"])
    s = s.squeeze(-1).masked_fill(mask.bool(), float("-inf"))                                # :256, :266-268
    return F.softmax(s, dim=-1), pooled, _mlp3_tanh64(w, "job_critic.", pooled, rnd)          # :278, :293


def _gat64(w, h1, h2):
    """GATLayer.forward (gat.py:82-159) on the 2-node graph [[1,1],[0,1]] of actor_critic.py:392-404: e = leaky_relu(s_i
    + t_j) (:73-80), node 1 attends to {1, 2}, node 2 to itself (softmax over one entry = 1)."""
    W, a = w["gat_layer.W"], w["gat_layer.a"]
    H = W.shape[0]
    t1, t2 = h1 @ W, h2 @ W                                                                      # gat.py:96
    a_s, a_d = a[0, :H, 0], a[0, H:, 0]
    e = F.leaky_relu(torch.stack((t1 @ a_s + t1 @ a_d, t1 @ a_s + t2 @ a_d), dim=-1), 0.2)
    att = torch.softmax(e, dim=-1)                                                              # gat.py:128
    return att[:, 0:1] * t1 + att[:, 1:2] * t2, t2                                              # gat.py:138


def f64_machine_trunk(w, fea1, fea2, groups):
    """actor_critic.py:381-444: two input projections, GAT x3 with ELU after the first two (:409-414), mean of the two
    node sets (:420), BatchNorm (:434), mean over machines (:444) -> nodes [B,M,H], pooled [B,H]."""
    B, M = fea1.shape[:2]
    h1 = F.linear(fea1.double(), w["m_fea_1_fcl.weight"]).reshape(B * M, -1)
    h2 = F.linear(fea2.double(), w["m_fea_2_fcl.weight"]).reshape(B * M, -1)
    h1, h2 = _gat64(w, h1, h2)
    h1, h2 = _gat64(w, F.elu(h1), F.elu(h2))
    h1, h2 = _gat64(w, F.elu(h1), F.elu(h2))
    nodes = _bn64((h1 + h2) / 2, w["bn.weight"], w["bn.bias"], groups).reshape(B, M, -1)
    return nodes, nodes.mean(dim=1)


def f64_machine_heads(w, nodes, pooled, h_pooled_o, mask):
    """actor_critic.py:459-498: m_policy over cat(node, pooled, h_pooled_o), x10 (:477), masked softmax; machine_critic."""
    x = torch.cat((nodes, pooled.unsqueeze(1).expand_as(nodes), h_pooled_o.unsqueeze(1).expand_as(nodes)), dim=-1)
    s = (_mlp3_tanh64(w, "m_policy.", x).squeeze(-1) * 10).masked_fill(mask.reshape(nodes.shape[:2]).bool(), float("-inf"))
    return F.softmax(s, dim=-1), _mlp3_tanh64(w, "machine_critic.", pooled)


def f64_critic(w, task_fea, A, fea1, fea2, groups):
    """Global_Critic_JointAction_GAT.forward (actor_critic.py:587-751): critic head on cat(pooled_m, pooled_o) (:737-750)."""
    pooled_o, _ = f64_graph_cnn(w, task_fea, A, groups)
    _, pooled_m = f64_machine_trunk(w, fea1, fea2, groups)
    return _mlp3_tanh64(w, "critic.", torch.cat((pooled_m, pooled_o), dim=-1))


def _golden_obs(g, s, J, M):
    """Observation of episode 0 before step s+1 of replay_j6m6_ls_esa.npz (s = -1: the initial state), as the env emits it."""
    B = g["t"].shape[0]
    if s < 0:
        tfea, adj, cand, mask, mfea2 = g["tfea0"][0], g["adj0"][0], np.tile(np.arange(J) * M, (B, 1)), np.zeros((B, J), bool), g["mfea20"][0]
    else:
        tfea, adj, cand, mask, mfea2 = g["tfea"][0, s], g["adj"][0, s], g["cand"][0, s], g["mask"][0, s], g["mfea2"][0, s]
    aw, asrc = tp.dense_to_ell(adj, M)
    return (torch.tensor(tfea, dtype=torch.float32).reshape(B, J * M, -1), torch.tensor(aw), torch.tensor(asrc), torch.tensor(cand.astype(np.int64)),
            torch.tensor(mask), torch.tensor(mfea2, dtype=torch.float32), torch.tensor(g["mfea1"][0, s + 1], dtype=torch.float32))


@pytest.mark.parametrize("H", [128, 32])
def test_fp64_restatement_forward_matches_reference_modules(H):
    """The restated forward against the reference modules' outputs (encoder_golden.npz), FP32 tolerance of test_encoder.py."""
    g = np.load(os.path.join(GOLD, "replay_j6m6_ls_esa.npz"))
    e = np.load(os.path.join(GOLD, "encoder_golden.npz"))
    J, M = int(g["J"]), int(g["M"])
    wj, wm = f64_params("job", H), f64_params("mch", H)
    close = lambda a, b, name: np.testing.assert_allclose(a.detach().numpy(), b, rtol=2e-4, atol=2e-5, err_msg=name)
    with torch.no_grad():
        for tag in ("init", "s05", "s20", "s34"):
            k = "H%d_%s_" % (H, tag)
            tfea, aw, asrc, cand, mask, mfea2, mfea1 = _golden_obs(g, int(e[k + "step"]), J, M)
            hgm = None if e[k + "hgm_in"].size == 0 else torch.tensor(e[k + "hgm_in"]).double()
            prob, pooled, jv = f64_job_evaluate(wj, tfea, ell_to_dense(aw, asrc), cand, hgm, mask, 1)
            close(prob, e[k + "prob"], "job prob " + tag)
            close(pooled, e[k + "pooled"], "job pooled " + tag)
            close(jv, e[k + "job_v"], "job value " + tag)
            nodes, pm = f64_machine_trunk(wm, mfea1, mfea2, 1)
            mp, mv = f64_machine_heads(wm, nodes, pm, torch.tensor(e[k + "pooled"]).double(), torch.tensor(e[k + "mmask"]))
            close(mp, e[k + "mch_prob"], "machine prob " + tag)
            close(pm, e[k + "mch_pooled"], "machine pooled " + tag)
            close(mv, e[k + "mch_v"], "machine value " + tag)


def _take(bt, name, idx):
    return bt.obs(name, idx) if hasattr(bt, "obs") and name in getattr(bt, "OBS", ()) else bt[name].index_select(0, idx)


def f64_minibatch_grads(bt, adv, idx, J, M, H, params, ge=None, eps=0.2, beta=0.01, pt=lambda t: t):
    """The PPO loss of one minibatch in float64 (ppo.py:214-296 = ppo_algorithm.py:716-1000), its gradients by autograd.
    Item i's job head gets item i-1's pooled machine embedding (not detached: the job loss reaches the machine actor),
    item 0 the learned `_input`; the surrogate and MSE terms are summed over (step, env) and divided by S*B.
    params: {net: f64 params}; pt: applied to the float64 observations (see _perturbation).  -> {net: {key: grad}}."""
    S, B, N = idx.numel(), bt["candidate"].shape[1], J * M
    G = S * (1 if ge is None else B // ge)
    wj, wm, wc = params["job"], params["mch"], params["crit"]
    d = lambda x: x.double()
    tf = pt(d(_take(bt, "task_fea", idx)).reshape(S * B, N, -1))
    A = pt(ell_to_dense(_take(bt, "adj_w", idx).reshape(S * B, N, 2), _take(bt, "adj_src", idx).reshape(S * B, N)))
    mf1 = pt(d(bt["mach_fea1"].index_select(0, idx)).reshape(S * B, M, 6))
    mf2 = pt(d(_take(bt, "mach_fea2", idx)).reshape(S * B, M, 8))
    nodes_m, pooled_m = f64_machine_trunk(wm, mf1, mf2, G)
    gm = torch.cat((wj["_input"][None, None, :].expand(1, B, H), pooled_m.reshape(S, B, H)[:-1]), dim=0).reshape(S * B, H)
    prob_j, pooled_o, job_v = f64_job_evaluate(wj, tf, A, bt["candidate"].index_select(0, idx).reshape(S * B, J), gm,
                                               bt["job_mask"].index_select(0, idx).reshape(S * B, J), G)
    prob_m, mch_v = f64_machine_heads(wm, nodes_m, pooled_m, pooled_o, bt["mach_mask"].index_select(0, idx).reshape(S * B, M))
    prob_j, prob_m, job_v, mch_v = prob_j.reshape(S, B, J), prob_m.reshape(S, B, M), job_v.reshape(S, B, 2), mch_v.reshape(S, B, 2)

    def logp_ent(prob, a):
        lp = torch.log(prob.gather(-1, a.long().unsqueeze(-1)).squeeze(-1))
        ent = -(prob * torch.log(torch.where(prob > 0, prob, torch.ones_like(prob)))).sum(-1)   # 0 log 0 = 0
        return lp, ent

    lpj, entj = logp_ent(prob_j, bt["a_job"].index_select(0, idx))
    lpm, entm = logp_ent(prob_m, bt["a_mach"].index_select(0, idx))
    rj = torch.exp(lpj - d(bt["log_a"].index_select(0, idx)))
    rm = torch.exp(lpm - d(bt["m_log_a"].index_select(0, idx)))
    ag, al = d(adv["adv_glob"].index_select(0, idx)), d(adv["adv_loc"].index_select(0, idx))
    tl, tg = d(adv["tgt_loc"].index_select(0, idx)), d(adv["tgt_glob"].index_select(0, idx))
    rw = d(bt["rw"].index_select(0, idx))
    wmk, wec, wtt = rw[..., 0], rw[..., 1], rw[..., 2]
    clip = lambda r, a: torch.min(r * a, torch.clamp(r, 1 - eps, 1 + eps) * a)
    glob = lambda r: wmk * clip(r, ag[..., 0]) + wec * (clip(r, ag[..., 1]) + clip(r, ag[..., 3])) + wtt * clip(r, ag[..., 2])
    loc_j = wmk * clip(rj, al[..., 0]) + wec * clip(rj, al[..., 3])
    loc_m = wec * clip(rm, al[..., 1]) + wtt * clip(rm, al[..., 2])
    sq = lambda a, b: ((a - b) ** 2).sum()
    crit_j = sq(wmk * job_v[..., 0], wmk * tl[..., 0]) + sq(wec * job_v[..., 1], wec * tl[..., 3])
    crit_m = sq(wec * mch_v[..., 0], wec * tl[..., 1]) + sq(wtt * mch_v[..., 1], wtt * tl[..., 2])
    inv = 1.0 / (S * B)
    lj = ((-2 * glob(rj) - loc_j - beta * entj).sum() + 0.5 * crit_j) * inv
    lm = ((-2 * glob(rm) - loc_m - beta * entm).sum() + 0.5 * crit_m) * inv
    out = {}
    ka, km = list(wj), list(wm)
    ga = torch.autograd.grad(lj + lm, [wj[k] for k in ka] + [wm[k] for k in km], allow_unused=True)
    out["job"] = dict(zip(ka, ga[:len(ka)]))
    out["mch"] = dict(zip(km, ga[len(ka):]))
    v = f64_critic(wc, tf, A, mf1, mf2, G).reshape(S, B, 4)
    lc = (sq(wmk * tg[..., 0], wmk * v[..., 0]) + sq(wec * tg[..., 1], wec * v[..., 1]) + sq(wec * tg[..., 3], wec * v[..., 3])
          + sq(wtt * tg[..., 2], wtt * v[..., 2])) * inv
    kc = list(wc)
    out["crit"] = dict(zip(kc, torch.autograd.grad(lc, [wc[k] for k in kc], allow_unused=True)))
    return out


def test_fp64_restatement_gradients_match_reference(monkeypatch):
    """The restated loss of the golden buffer's first minibatch, on the advantages `MAPPOUpdate.advantages` computes, against
    the reference's gradients -- the same tolerance as the device path."""
    _kernel_restatements(monkeypatch)
    _, (bt, adv, idx, J, M, H) = _first_minibatch_device(torch.device("cpu"))
    grads = f64_minibatch_grads(bt, adv, idx, J, M, H, {t: f64_params(t, H) for t in NETS})
    for tag in NETS:
        fails, _ = compare_grads(grads[tag], _golden_grads(tag))
        assert not fails, (tag, fails)


# ---- part 3: device gradients against the FP64 restatement (gpu) ----------------------------------------------------
def _states(J, M, E, B, S, edge, seed=7):
    """S consecutive states of B envs under the random policy, stacked to S*B envs: observations before each step, the
    candidate-machine features of the op drawn at that step."""
    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    d = ins.reference_stream_instances(B, J, M, E, seed) if edge else ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed))
    env.obs()
    keys = ("task_fea", "adj_w", "adj_src", "job_mask", "candidate", "mach_fea")
    out = {k: [] for k in keys + ("mfea1", "mach_mask")}
    for _ in range(S):
        for k in keys:
            out[k].append(getattr(env, k).clone())
        env.random_step(seed=seed)
        out["mfea1"].append(env.mfea1_buf.clone())
        out["mach_mask"].append(env.mach_mask.clone())
    return {k: torch.cat(v, dim=0) for k, v in out.items()}


SHAPES = [  # J, M, E, B, ge, S, edge instances
    (6, 6, 2, 32, 16, 36, False), (6, 6, 2, 32, None, 36, False), (10, 10, 3, 16, 8, 12, False), (30, 20, 5, 4, 4, 6, False),
    (1, 64, 7, 8, 4, 64, True), (48, 64, 4, 2, 2, 2, True)]
_ids = lambda s: "J%dM%dE%d_B%d_ge%s_S%d" % s[:6]

# Rounding of the device path against the conditioning of each gradient.  A plain relative bound cannot tell a kernel error
# from an ill-conditioned gradient: the critic's only cotangent reaches its machine trunk through the env means of one
# BatchNorm group (pooled_m), whose backward subtracts the group mean of that cotangent and its projection on xhat, and at
# J1M64 with 4-env groups what is left is ~1e-3 of the terms.  So every comparison against FP64 also measures how far the
# FP64 gradient itself moves when its inputs and weights are perturbed at the working precision's unit roundoff
# (relative u = 2^-24 for FP32, 2^-11 for the TF32 operands): `sens`, the larger of two such perturbations.  A tensor
# passes when its error is within FLOOR or within K x sens.  A kernel error of the size a gradient itself has would
# show as an error far above its sens; a rounding effect stays within a small multiple of it.
U_FP32, U_TF32 = 2.0 ** -24, 2.0 ** -11


def _perturbation(eps, seed, dev):
    """t -> t * (1 + eps * r), r uniform in [-1, 1] elementwise (zeros stay zero: the adjacency keeps its pattern)."""
    if eps == 0:
        return lambda t: t
    gen = torch.Generator(device=dev).manual_seed(seed)
    return lambda t: t * (1 + eps * (2 * torch.rand(t.shape, generator=gen, device=dev, dtype=torch.float64) - 1))


def _perturbed_params(sds, H, pt, dev):
    return {t: {k: pt(v.detach()).detach().requires_grad_(True) for k, v in f64_params(t, H, sd=sds[t], device=dev).items()}
            for t in NETS}


def _f64_vjps(st, sds, G, H, hgm, hpo, cots, pt):
    """FP64 VJPs of the three networks on (perturbed) inputs and weights -> {net: {key: grad}}."""
    w64 = _perturbed_params(sds, H, pt, hgm.device)
    A = pt(ell_to_dense(st["adj_w"], st["adj_src"]))
    tf, mf1, mf2 = pt(st["task_fea"].double()), pt(st["mfea1"].double()), pt(st["mach_fea"].double())
    res = {}
    x64 = pt(hgm.double()).requires_grad_(True)
    outs = f64_job_evaluate(w64["job"], tf, A, st["candidate"], x64, st["job_mask"], G)
    ks = list(w64["job"])
    gr = torch.autograd.grad(outs, [w64["job"][k] for k in ks] + [x64], cots["job"], allow_unused=True)
    res["job"] = dict(zip(ks + ["h_g_m_pooled"], gr))
    x64 = pt(hpo.double()).requires_grad_(True)
    n64, p64 = f64_machine_trunk(w64["mch"], mf1, mf2, G)
    pr64, mv64 = f64_machine_heads(w64["mch"], n64, p64, x64, st["mach_mask"])
    ks = list(w64["mch"])
    gr = torch.autograd.grad((pr64, p64, mv64), [w64["mch"][k] for k in ks] + [x64], cots["mch"], allow_unused=True)
    res["mch"] = dict(zip(ks + ["h_pooled_o"], gr))
    v64 = f64_critic(w64["crit"], tf, A, mf1, mf2, G)
    ks = list(w64["crit"])
    res["crit"] = dict(zip(ks, torch.autograd.grad(v64, [w64["crit"][k] for k in ks], cots["crit"], allow_unused=True)))
    return res


def _sensitivity(ref, perturbed):
    """{key: largest relative move of the FP64 gradient over the perturbed runs}."""
    out = {}
    for k, r in ref.items():
        if r is None:
            continue
        rn = float(r.double().norm())
        out[k] = max(float((p[k].double() - r.double()).norm()) / rn for p in perturbed) if rn > 0 else 0.0
    return out


def check_conditioned(got, ref, sens, floor, k_sens, zero_tol, cos_min=None, encoder_floor=None):
    """compare_grads with a per-tensor bound max(floor, k_sens * sens[key]) on the relative error, and cosine >= cos_min
    where given and the tensor is not noise-level at the working precision (sens < 0.1).  encoder_floor: the floor of the
    graph-encoder tensors (FP32 path, see FP32_ENCODER_FLOOR).  -> (failures, {key: (rel, cos, sens)})."""
    fails, stats = [], {}
    for key, rv in ref.items():
        if rv is not None and (_zero_grad_bias(key) or float(rv.abs().max()) == 0.0):
            continue                                             # _zero_bounded
        fl = encoder_floor if encoder_floor is not None and key.startswith("encoder.") else floor
        b = max(fl, k_sens * sens.get(key, 0.0))
        f, st = compare_grads({key: got.get(key)}, {key: rv}, rel=b, a=b, r=b, zero_tol=zero_tol)
        fails += f
        if key in st:
            stats[key] = st[key] + (sens.get(key, 0.0),)
            if cos_min is not None and sens.get(key, 0.0) < 0.1 and not math.isnan(st[key][1]) and st[key][1] < cos_min:
                fails.append((key, "cosine %.6f" % st[key][1]))
    return fails, stats


def _zero_bounded(got, ref, zero_tol):
    """The zero-gradient tensors (see _zero_grad_bias) of one network against the norm of its other gradients."""
    norm = math.sqrt(sum(float((v.double() ** 2).sum()) for k, v in ref.items() if v is not None))
    bad = []
    for k, v in ref.items():
        if v is not None and (_zero_grad_bias(k) or float(v.abs().max()) == 0.0) and \
                float((got[k].double() - v.double()).norm()) > zero_tol * norm:
            bad.append((k, "zero-gradient tensor off by %.3g of the network norm" % (float((got[k].double() - v.double()).norm()) / norm)))
    return bad


def _report(tag, label, stats):
    worst = max(stats.items(), key=lambda kv: kv[1][0])
    ratio = max((v[0] / v[2] for v in stats.values() if v[2] > 0), default=0.0)
    cmin = min((v[1] for v in stats.values() if not math.isnan(v[1])), default=float("nan"))
    print("%s %s worst rel %.3g (%s, sens %.3g), min cos %.7f, worst rel/sens %.3g"
          % (label, tag, worst[1][0], worst[0], worst[1][2], cmin, ratio))


def _vjp_case(J, M, E, B, ge, S, edge, tf32):
    """Device VJPs of the three networks (FP32 path, or the tcgen05 path with tf32) and the FP64 ones on the same states
    and random cotangents -> {net: (device grads, FP64 grads, sens)}."""
    dev = torch.device("cuda", 0)
    H = 128
    st = _states(J, M, E, B, S, edge)
    R = S * B
    G = S if ge is None else R // ge
    gen = torch.Generator(device=dev).manual_seed(J * 100 + M)
    sds = {t: enc.seeded_state_dict(KEYS[t](H), SEEDS[t]) for t in NETS}
    job = enc.JobActor(sds["job"], J, M, hidden=H, trainable=True)
    mch = enc.MachineActor(sds["mch"], M, hidden=H, trainable=True)
    crit = enc.GlobalCritic(sds["crit"], J, M, hidden=H, trainable=True)
    for n in (job, mch, crit):
        n.train_tf32 = tf32
    hgm = torch.randn(R, H, device=dev, generator=gen)
    hpo = torch.randn(R, H, device=dev, generator=gen)
    got, cots = {}, {}
    x = hgm.clone().requires_grad_(True)
    outs = job.evaluate(st["task_fea"], st["adj_w"], st["adj_src"], st["candidate"], x, st["job_mask"], groups=G)
    cots["job"] = [torch.randn(o.shape, device=dev, generator=gen, dtype=torch.float64) for o in outs]
    torch.autograd.backward(list(outs), [c.float() for c in cots["job"]])
    got["job"] = _net_grads(job); got["job"]["h_g_m_pooled"] = x.grad
    x = hpo.clone().requires_grad_(True)
    nodes, pooled = mch.trunk(st["mfea1"], st["mach_fea"], groups=G)
    prob, mv = mch.heads(nodes, pooled, x, st["mach_mask"])
    cots["mch"] = [torch.randn(o.shape, device=dev, generator=gen, dtype=torch.float64) for o in (prob, pooled, mv)]
    torch.autograd.backward([prob, pooled, mv], [c.float() for c in cots["mch"]])
    got["mch"] = _net_grads(mch); got["mch"]["h_pooled_o"] = x.grad
    v = crit.forward(st["task_fea"], st["adj_w"], st["adj_src"], st["mfea1"], st["mach_fea"], groups=G)
    cots["crit"] = torch.randn(v.shape, device=dev, generator=gen, dtype=torch.float64)
    v.backward(cots["crit"].float())
    got["crit"] = _net_grads(crit)
    ref = _f64_vjps(st, sds, G, H, hgm, hpo, cots, _perturbation(0, 0, dev))
    eps = U_TF32 if tf32 else U_FP32
    pert = [_f64_vjps(st, sds, G, H, hgm, hpo, cots, _perturbation(eps, 100 + i, dev)) for i in (0, 1)]
    return {t: (got[t], ref[t], _sensitivity(ref[t], [p[t] for p in pert])) for t in NETS}


# Measured on an NVIDIA B200 (1000 W), largest error / sens over the network VJP and whole-minibatch cases:
#   FP32 path, every tensor outside the graph encoders: 27 (worst error 8.5e-5).  The critic's machine trunk at J1M64
#     (gat_layer.a 3.5e-3, m_fea_2_fcl 2.5e-3, gat_layer.W 2.3e-3 where the machine actor's trunk is at 1.9e-5) is
#     conditioning: the FP64 gradient itself moves by 3.0e-3 under an FP32-sized perturbation, ratio 2.4.
#   TF32 path, every tensor: 1.7.  The critic's gat_layer.a (0.24, cosine 0.980) and m_fea_2_fcl (0.197) at J6M6 have
#     sens 0.21 and 0.17: the critic's trunk gradient is that ill-conditioned, not a kernel error; at J1M64 it is noise
#     (sens > 1, cosines down to 0.89), so the cosine bound skips tensors with sens >= 0.1.
#   FP32 graph encoders: not explained by conditioning (error / sens up to 3.7e3, worst error 1.05e-2 for the critic at
#     J6M6 with one group per step).  The FP32 neighbourhood mean is the cause -- formed in FP64 as the reference does
#     (gcn_mlp.py:125) the golden minibatch goes from 1.4e-3 to 5.5e-6 -- but not its final rounding: the FP64 network
#     with its mean rounded to FP32 moves by 1.7e-7 only.  What amplifies the FP32 sum's own rounding is open; those
#     tensors keep FP32_ENCODER_FLOOR, about 3x the measured worst.
FP32_FLOOR, FP32_K, FP32_ENCODER_FLOOR = 1e-4, 30.0, 3e-2
TF32_FLOOR, TF32_K, TF32_COS = 1e-3, 5.0, 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_ids)
def test_network_vjps_match_fp64_restatement(shape):
    """Parameter gradients and the cross-network inputs' gradients of each network under random output cotangents, FP32
    path against the FP64 restatement, within FP32_FLOOR or FP32_K times the tensor's FP64 sensitivity to FP32 rounding."""
    res = _vjp_case(*shape, tf32=False)
    bad = []
    for tag in NETS:
        got, ref, sens = res[tag]
        fails, stats = check_conditioned(got, ref, sens, FP32_FLOOR, FP32_K, zero_tol=1.0, encoder_floor=FP32_ENCODER_FLOOR)
        fails += _zero_bounded(got, ref, 1e-4)
        _report(tag, "fp32 %s" % _ids(shape), stats)
        bad += [(tag,) + f for f in fails]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [SHAPES[0], SHAPES[2], SHAPES[4]], ids=_ids)
def test_network_vjps_tcgen05_path_against_fp64(shape):
    """The tcgen05 TF32 training path (PPOConfig.encoder_tf32) against FP64, bounded by the tensor's FP64 sensitivity to a
    perturbation at the TF32 unit roundoff."""
    res = _vjp_case(*shape, tf32=True)
    bad = []
    for tag in NETS:
        got, ref, sens = res[tag]
        fails, stats = check_conditioned(got, ref, sens, TF32_FLOOR, TF32_K, zero_tol=1.0, cos_min=TF32_COS)
        fails += _zero_bounded(got, ref, 1e-2)
        _report(tag, "tf32 %s" % _ids(shape), stats)
        for k, (e, c, sn) in sorted(stats.items(), key=lambda kv: -kv[1][0])[:4]:
            print("   ", k, "rel %.3g cos %.6f sens %.3g" % (e, c, sn))
        bad += [(tag,) + f for f in fails]
    assert not bad, bad


def _buffer(J, M, E, B, ge, seed=5):
    """One FP32 episode of B envs with bn_group_envs = ge -> RolloutBuffer (the training path's own buffer)."""
    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    rom = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(128), SEEDS["job"]), J, M)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), SEEDS["mch"]), M)
    ro = rom.Rollout(env, job, mch, greedy=False, seed=3, bn_group_envs=ge)
    return ppo.collect(ro, [ins.random_weights(0, B, seed)])


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2, 32, 16), (10, 10, 3, 16, 8)], ids=lambda s: "J%dM%dE%d_B%d_ge%d" % s)
@pytest.mark.parametrize("chunked", [False, True], ids=["one_chunk", "chunks_of_7_steps"])
@pytest.mark.parametrize("tf32", [False, True], ids=["fp32", "tcgen05"])
def test_minibatch_gradients_match_fp64_loss(size, chunked, tf32):
    """Whole `_minibatch` (lr 0, no clipping) on a buffer from `ppo.collect`, one minibatch of the episode's N steps in a
    shuffled order, against the FP64 restated loss on the same advantages.  chunks_of_7_steps sets max_rows so that the
    minibatch is walked in gradient-accumulation chunks of 7 steps: the machine trunk's one-step overlap with the previous
    chunk and the adj_dst the critic pass reuses from the actor pass are on the path."""
    J, M, E, B, ge = size
    N, H = J * M, 128
    dev = torch.device("cuda", 0)
    bt = _buffer(J, M, E, B, ge)
    sds = {t: enc.seeded_state_dict(KEYS[t](H), SEEDS[t]) for t in NETS}
    job = enc.JobActor(sds["job"], J, M, hidden=H, trainable=True)
    mch = enc.MachineActor(sds["mch"], M, hidden=H, trainable=True)
    crit = enc.GlobalCritic(sds["crit"], J, M, hidden=H, trainable=True)
    up = ppo.MAPPOUpdate(job, mch, crit, ppo.PPOConfig(lr=0.0, use_grad_clip=False, bn_group_envs=ge, encoder_tf32=tf32),
                         max_rows=7 * B * N if chunked else 1 << 21)
    cs = up._steps_per_chunk(max(1, min(N, up.max_rows // (B * N))), B, extra=1)
    assert (cs == 7) if chunked else (cs == N)
    with torch.no_grad():
        adv = up.advantages(bt)
    idx = torch.randperm(N, generator=torch.Generator().manual_seed(J)).to(dev)
    up._minibatch(bt, adv, idx)
    got = {"job": _net_grads(job), "mch": _net_grads(mch), "crit": _net_grads(crit)}
    runs = []
    for i, eps in enumerate((0.0, U_TF32 if tf32 else U_FP32, U_TF32 if tf32 else U_FP32)):
        pt = _perturbation(eps, 200 + i, dev)
        runs.append(f64_minibatch_grads(bt, adv, idx, J, M, H, _perturbed_params(sds, H, pt, dev), ge=ge, pt=pt))
    bad = []
    for tag in NETS:
        sens = _sensitivity(runs[0][tag], [r[tag] for r in runs[1:]])
        if tf32:
            fails, stats = check_conditioned(got[tag], runs[0][tag], sens, TF32_FLOOR, TF32_K, zero_tol=1.0, cos_min=TF32_COS)
            fails += _zero_bounded(got[tag], runs[0][tag], 1e-2)
        else:
            fails, stats = check_conditioned(got[tag], runs[0][tag], sens, FP32_FLOOR, FP32_K, zero_tol=1.0,
                                                 encoder_floor=FP32_ENCODER_FLOOR)
            fails += _zero_bounded(got[tag], runs[0][tag], 1e-4)
        _report(tag, "minibatch %s %s %s" % (size, "chunked" if chunked else "one chunk", "tf32" if tf32 else "fp32"), stats)
        bad += [(tag,) + f for f in fails]
    assert not bad, bad


# ---- part 4: the training kernels at their edges (gpu) --------------------------------------------------------------
def _bn_ref(x, w, b, gy, G, relu, mask=None):
    """FP64 autograd of BatchNorm (+ReLU).  mask: the ReLU decisions to back-propagate through (default: FP64's own)."""
    x2, w2, b2 = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    xs = x2.reshape(G, -1, x.shape[-1])
    var, mean = torch.var_mean(xs, dim=1, unbiased=False, keepdim=True)
    y = ((xs - mean) * torch.rsqrt(var + 1e-5) * w2 + b2).reshape(x.shape)
    if relu:
        y = y * ((y > 0) if mask is None else mask).double()
    y.backward(gy.double())
    return y.detach(), x2.grad, w2.grad, b2.grad


@pytest.mark.gpu
@pytest.mark.parametrize("R", [96, 576])
@pytest.mark.parametrize("offset", [0, 30, 100, 1000])
@pytest.mark.parametrize("relu", [False, True])
def test_batchnorm_kernels_with_large_column_means(R, offset, relu):
    """Rows per group of the trainer (16 envs x 6 machines, 16 envs x 36 ops), C = 128, column means of `offset` standard
    deviations: forward and backward against FP64 autograd.

    Tolerance 2e-4 (test_ppo.py's BatchNorm test) plus 8 * offset * 2^-24: the mean is handed to the apply and backward
    passes as an FP32 number, so it carries a rounding error of up to offset * 2^-24 standard deviations, which shifts
    every xhat by that much (dgamma / dbeta: times sqrt(G*R), see below).  The backward is compared given the kernel's own ReLU decisions (an element with y within
    rounding of 0 may fall on either side; that choice is the forward's, checked through y).  With the statistics summed
    as x^2 - mean^2 every case from 30 standard deviations failed 2e-4 (relative rstd errors of 5e-5 to 5e-2 in
    emulation); summed about the group's first row they pass."""
    dev = torch.device("cuda", 0)
    G, C = 8, 128
    gen = torch.Generator(device=dev).manual_seed(R + offset)
    std = torch.rand(C, device=dev, generator=gen) + 0.5
    mu = offset * std * torch.sign(torch.randn(C, device=dev, generator=gen))
    x = torch.randn(G * R, C, device=dev, generator=gen) * std + mu
    w = torch.rand(C, device=dev, generator=gen) + 0.5
    b = torch.randn(C, device=dev, generator=gen) * 0.3
    gy = torch.randn(G * R, C, device=dev, generator=gen)
    y, mean, rstd = enc.bn_forward(x, w, b, 1e-5, G, relu)
    dx, dw, db = enc.bn_backward(x, gy, w, b, mean, rstd, G, relu)
    ry = _bn_ref(x, w, b, gy, G, relu)[0]
    _, rdx, rdw, rdb = _bn_ref(x, w, b, gy, G, relu, mask=(y > 0) if relu else None)
    tol = 2e-4 + 8 * offset * 2.0 ** -24
    for a, r, name in ((y, ry, "y"), (dx, rdx, "dx")):
        np.testing.assert_allclose(a.double().cpu().numpy(), r.cpu().numpy(), rtol=tol, atol=tol, err_msg=name)
    # dgamma = sum of gy * xhat over the G*R rows: the mean's rounding is one shift per column, so it adds up as sqrt(G*R)
    tol_sum = 2e-4 + 8 * offset * 2.0 ** -24 * (G * R) ** 0.5
    for a, r, name in ((dw, rdw, "dgamma"), (db, rdb, "dbeta")):
        np.testing.assert_allclose(a.double().cpu().numpy(), r.cpu().numpy(), rtol=2e-4, atol=tol_sum, err_msg=name)


@pytest.mark.gpu
def test_batchnorm_kernels_at_the_group_limit():
    """G = 65,535 groups (the grid.y limit) of 3 rows; G = 65,536 is refused with MTFJSP_E_ARG."""
    lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
    dev = torch.device("cuda", 0)
    G, R, C = 65535, 3, 8
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(G * R, C, device=dev, generator=gen) * 2 + 1
    w = torch.rand(C, device=dev, generator=gen) + 0.5
    b = torch.randn(C, device=dev, generator=gen) * 0.3
    gy = torch.randn(G * R, C, device=dev, generator=gen)
    y, mean, rstd = enc.bn_forward(x, w, b, 1e-5, G, True)
    dx, dw, db = enc.bn_backward(x, gy, w, b, mean, rstd, G, True)
    ry, rdx, rdw, rdb = _bn_ref(x, w, b, gy, G, True)
    for a, r, name in ((y, ry, "y"), (dx, rdx, "dx")):
        np.testing.assert_allclose(a.double().cpu().numpy(), r.cpu().numpy(), rtol=2e-4, atol=2e-4, err_msg=name)
    for a, r, name in ((dw, rdw, "dgamma"), (db, rdb, "dbeta")):      # sums over 196,605 rows
        np.testing.assert_allclose(a.double().cpu().numpy(), r.cpu().numpy(), rtol=2e-4, atol=2e-4 * R * G ** 0.5, err_msg=name)
    G = 65536
    x = torch.zeros(G * R, C, device=dev)
    y, m, r = torch.empty_like(x), torch.empty(G, C, device=dev), torch.empty(G, C, device=dev)
    ws = torch.empty(G, 2, C, dtype=torch.float64, device=dev)
    P = enc._ptr
    rc = lib.lib().mtfjsp_enc_bn_fwd(P(x), P(w), P(b), 1e-5, G, R, C, 0, P(y), P(m), P(r), P(ws), enc._stream())
    assert rc == -1  # MTFJSP_E_ARG
    rc = lib.lib().mtfjsp_enc_bn_bwd(P(x), P(x), P(w), P(b), P(m), P(r), G, R, C, 0, P(y), P(ws), enc._stream())
    assert rc == -1


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2, 32), (10, 10, 3, 16), (30, 20, 5, 4), (1, 64, 7, 8), (48, 64, 4, 2), (1678, 2, 1, 2)],
                         ids=lambda s: "J%dM%dE%d" % s[:3])
@pytest.mark.parametrize("C", [12, 128])
def test_aggregation_forward_and_backward_on_real_adjacency(size, C):
    """aggregate + its backward (with ell_invert) on the ELL adjacency half-way through random episodes, against the dense
    FP64 product and its transpose: within 3 FP32 ulp of the magnitude sum forward (as test_encoder.py), 4 backward (the
    weight is multiplied by the rounded 1/deg before the fused multiply-add)."""
    J, M, E, B = size
    edge = (J, M) in ((1, 64), (48, 64), (1678, 2))
    st = _states(J, M, E, B, max(1, (J * M) // 2), edge)
    aw, asrc = st["adj_w"][-B:].contiguous(), st["adj_src"][-B:].contiguous()
    N = J * M
    assert bool((asrc >= 0).any()) and bool((aw[..., 0] != 0).any())
    A = ell_to_dense(aw, asrc)
    deg = (A != 0).sum(-1, keepdim=True).double()
    gen = torch.Generator(device="cuda").manual_seed(C + N)
    h = torch.randn(B, N, C, device="cuda", generator=gen).requires_grad_(True)
    g = torch.randn(B, N, C, device="cuda", generator=gen)
    out = enc.aggregate(h, aw, asrc, adj_dst=enc.ell_invert(asrc))
    out.backward(g)
    ulp = 2.0 ** -24
    ref = torch.bmm(A, h.detach().double()) / deg
    bound = 3 * ulp * torch.bmm(A.abs(), h.detach().double().abs()) / deg + 1e-30
    assert bool(((out.detach().double() - ref).abs() <= bound).all()), float(((out.detach().double() - ref).abs() / bound).max())
    rg = torch.bmm(A.transpose(1, 2), g.double() / deg)
    gb = 4 * ulp * torch.bmm(A.abs().transpose(1, 2), g.double().abs() / deg) + 1e-30
    assert bool(((h.grad.double() - rg).abs() <= gb).all()), float(((h.grad.double() - rg).abs() / gb).max())
    print("aggregation", size, C, "worst error in ulp of the magnitude sum: forward %.2f, backward %.2f" % (
        3 * float(((out.detach().double() - ref).abs() / bound).max()), 4 * float(((h.grad.double() - rg).abs() / gb).max())))


@pytest.mark.gpu
@pytest.mark.parametrize("R", [3 * 9472 + 5, 221184])
@pytest.mark.parametrize("mode", [1, 2])
def test_gat_attend_backward_over_the_grid_stride_loop(R, mode):
    """R above the 1,184 blocks x 8 warps of the backward's grid, so every warp accumulates several rows; against FP64."""
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(R + mode)
    t0 = torch.randn(2 * R, 128, device=dev, generator=gen)
    as0 = torch.randn(128, device=dev, generator=gen) * 0.1
    ad0 = torch.randn(128, device=dev, generator=gen) * 0.1
    gy = torch.randn(R if mode == 2 else 2 * R, 128, device=dev, generator=gen)
    t, a, b = (v.clone().requires_grad_(True) for v in (t0, as0, ad0))
    enc.gat_attend_train(t, a, b, mode).backward(gy)
    t2, a2, b2 = (v.double().requires_grad_(True) for v in (t0, as0, ad0))
    wd = {"gat_layer.W": torch.eye(128, dtype=torch.float64, device=dev), "gat_layer.a": torch.cat((a2, b2))[None, :, None]}
    h1, h2 = _gat64(wd, t2[:R], t2[R:])
    y = torch.stack((h1, h2), 1).mean(1) if mode == 2 else torch.cat((F.elu(h1), F.elu(h2)), 0)
    y.backward(gy.double())
    np.testing.assert_allclose(t.grad.double().cpu().numpy(), t2.grad.cpu().numpy(), rtol=0, atol=2e-4, err_msg="dt")
    for x, r, name in ((a.grad, a2.grad, "da_src"), (b.grad, b2.grad, "da_dst")):
        rel = float((x.double() - r).norm() / r.norm())
        assert rel < 1e-4, (name, rel)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 32])
@pytest.mark.parametrize("greedy", [True, False])
def test_selection_kernel_at_one_and_thirty_two_entries(R, greedy):
    """enc.select at R = 1 (the job head at J = 1) and R = 32 (every lane): probabilities and the log-probability of the
    chosen entry (the update's log_a) against FP64."""
    dev = torch.device("cuda", 0)
    B = 4099
    gen = torch.Generator(device=dev).manual_seed(R)
    s = torch.randn(B, R, device=dev, generator=gen) * 3
    mask = (torch.rand(B, R, device=dev, generator=gen) < 0.3).to(torch.uint8)
    mask[:, 0] = 0                                                     # every env keeps an open entry
    counter = torch.zeros((), dtype=torch.int64, device=dev)
    prob, a, la, task = enc.select(s, mask, None, 1.0, greedy, (5, counter), 0)
    ref = torch.softmax(s.double().masked_fill(mask.bool(), float("-inf")), -1)
    np.testing.assert_allclose(prob.double().cpu().numpy(), ref.cpu().numpy(), rtol=2e-6, atol=1e-7)
    assert bool((mask.gather(1, a[:, None]) == 0).all())
    np.testing.assert_allclose(la.double().cpu().numpy(), torch.log(ref.gather(1, a[:, None])[:, 0]).cpu().numpy(), rtol=1e-5, atol=1e-6)
    if greedy:
        assert torch.equal(a, s.masked_fill(mask.bool(), float("-inf")).argmax(-1))
    if R == 1:
        assert bool((a == 0).all()) and bool((la == 0).all())
