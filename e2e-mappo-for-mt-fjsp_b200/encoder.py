"""GNN encoder + actor heads of the MAPPO rollout on the device (SURVEY.md 8 a13).

Forward-only mirrors of the reference networks that consume the environment's native observation layout directly
(compact ELL adjacency, F32 feature rows), with the reference's state_dict key names so shipped checkpoints load:

    JobActor      <- model/actor_critic.py:26-296   Operation_Actor_JointAction_selfCritic
                     (GIN-style encoder model/gcn_mlp.py:109-197, 204-249; MLPActor / MLPCritic :322-434)
    MachineActor  <- model/actor_critic.py:299-498  Machine_Actor_JointAction_selfGAT_selfCritic
                     (GAT layer model/gat.py:68-159 over the fixed 2-node graph [[1,1],[0,1]])
    EsaJobActor, EsaMachineActor <- model/actor_critic.py:945-1404  esa_Operation_Actor_Critic, esa_Machine_Actor
                     (the ESA-PPO baseline the reference's test table compares against; inference only)

What runs where (round 1): the neighbour aggregation (reference: dense adj -> COO -> FP64 cuSPARSE SpMM -> second
SpMM for the degree) is the hand-written `mtfjsp_enc_aggregate` kernel over ELL; graph pooling is
`mtfjsp_enc_graph_mean`; the 2x2 GAT attention is closed-form elementwise math; the dense per-node projections run
on the tcgen05 kernel `mtfjsp_enc_linear_tf32` with `precision="tf32"` (BatchNorm statistics in its epilogue, the
folded BatchNorm + ReLU of the previous layer in its prologue; per-env statistics and per-group affines with groups > 1,
the *_grouped entry points) or on library FP32 GEMMs with `precision="fp32"`;
BatchNorm uses batch statistics exactly as the reference does (its modules are never put in eval mode, SURVEY.md 3.3).
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from ._lib import check


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _optr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _aggregate_raw(h, adj_w, adj_src, in_scale=None, in_shift=None, relu=False):
    B, N, Cc = h.shape
    h = h.contiguous()
    out = torch.empty_like(h)
    if in_scale is not None and in_scale.dim() == 2:  # per-group affine [G,C] (grouped BatchNorm)
        check(_lib.lib().mtfjsp_enc_aggregate_grouped(_ptr(h), _ptr(adj_w), _ptr(adj_src), _ptr(out), B, N, Cc, _ptr(in_scale),
                                                      _ptr(in_shift), int(relu), B // in_scale.shape[0], _stream()),
              "mtfjsp_enc_aggregate_grouped")
        return out
    check(_lib.lib().mtfjsp_enc_aggregate(_ptr(h), _ptr(adj_w), _ptr(adj_src), _ptr(out), B, N, Cc, _optr(in_scale),
                                          _optr(in_shift), int(relu), _stream()), "mtfjsp_enc_aggregate")
    return out


def ell_invert(adj_src):
    """adj_dst[b,u] = v with adj_src[b,v] == u (machine successor), -1 if none; needed by the aggregation backward."""
    B, N = adj_src.shape
    adj_dst = torch.empty_like(adj_src)
    check(_lib.lib().mtfjsp_enc_ell_invert(_ptr(adj_src.contiguous()), _ptr(adj_dst), B, N, _stream()), "mtfjsp_enc_ell_invert")
    return adj_dst


class _AggregateFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, adj_w, adj_src, adj_dst):
        ctx.save_for_backward(adj_w, adj_src, adj_dst)
        return _aggregate_raw(h, adj_w, adj_src)

    @staticmethod
    def backward(ctx, g):
        adj_w, adj_src, adj_dst = ctx.saved_tensors
        B, N, Cc = g.shape
        g = g.contiguous()
        out = torch.empty_like(g)
        check(_lib.lib().mtfjsp_enc_aggregate_bwd(_ptr(g), _ptr(adj_w), _ptr(adj_src), _ptr(adj_dst), _ptr(out), B, N, Cc,
                                                  _stream()), "mtfjsp_enc_aggregate_bwd")
        return out, None, None, None


def aggregate(h, adj_w, adj_src, in_scale=None, in_shift=None, relu=False, adj_dst=None):
    """out[b,v] = (x[b,v] + w_job*x[b,v-1] + w_mach*x[b,src]) / in_degree (FP32 FMAs); h [B,N,C] f32;
    x = relu?(h*in_scale+in_shift) when an input affine is given (the producing layer's BatchNorm, folded in).
    Differentiable in h (PPO update): the backward is the transposed gather, `mtfjsp_enc_aggregate_bwd`."""
    adj_w, adj_src = adj_w.contiguous(), adj_src.contiguous()
    if torch.is_grad_enabled() and h.requires_grad:
        if in_scale is not None:
            raise ValueError("the folded input affine is an inference-path option")
        return _AggregateFn.apply(h, adj_w, adj_src, ell_invert(adj_src) if adj_dst is None else adj_dst)
    return _aggregate_raw(h, adj_w, adj_src, in_scale, in_shift, relu)


class _GraphMeanFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h):
        ctx.N = h.shape[1]
        return _graph_mean_raw(h)

    @staticmethod
    def backward(ctx, g):
        inv = torch.tensor(1.0 / ctx.N, dtype=torch.float32).item()
        return (g * inv).unsqueeze(1).expand(-1, ctx.N, -1)


def aggregate_linear_tf32(h, adj_w, adj_src, weight, bias, in_scale=None, in_shift=None, relu=False, stats=None):
    """mtfjsp_enc_aggregate_linear_tf32: aggregate(h) followed by the layer's product, in one launch (the weighted
    neighbourhood mean is applied to the product rows in the epilogue).  h [B,N,128] -> [B*N,128], or None when this
    form is not available for the size (the caller then runs aggregate + linear_tf32)."""
    B, N = h.shape[0], h.shape[1]
    if N > 128 or h.shape[2] != 128:
        return None
    z = torch.empty((B * N, 128), dtype=torch.float32, device=h.device)
    rc = _lib.lib().mtfjsp_enc_aggregate_linear_tf32(_ptr(h), B, N, _ptr(adj_w), _ptr(adj_src), _ptr(weight), _optr(bias),
                                                     _optr(in_scale), _optr(in_shift), 1 if relu else 0, _ptr(z), _optr(stats),
                                                     _stream())
    if rc == -3:  # MTFJSP_E_STATE: this form is not available here (driver without the TMA entry point)
        return None
    check(rc, "mtfjsp_enc_aggregate_linear_tf32")
    return z


def select(scores, mask, cand, scale, greedy, rng, stream_id):
    """mtfjsp_enc_select: masked softmax, one draw (or the arg-max), its log-probability and the candidate behind it in one
    launch.  scores [B,R] f32, mask [B,R] u8 / bool (1 = excluded), cand [B,R] i32 or None, rng = (seed, counter) with
    counter a device int64 tensor the caller advances once per step -> prob [B,R], action [B] i64, log_a [B], task [B] i64."""
    B, R = scores.shape
    dev = scores.device
    prob = torch.empty((B, R), dtype=torch.float32, device=dev)
    action = torch.empty(B, dtype=torch.int64, device=dev)
    log_a = torch.empty(B, dtype=torch.float32, device=dev)
    task = torch.empty(B, dtype=torch.int64, device=dev)
    m8 = mask.reshape(B, R)
    m8 = (m8 if m8.dtype == torch.uint8 else m8.to(torch.uint8)).contiguous()
    seed, counter = rng if rng is not None else (0, None)
    check(_lib.lib().mtfjsp_enc_select(_ptr(scores.contiguous()), _ptr(m8), _optr(cand), float(scale), R, B, 1 if greedy else 0,
                                       int(seed) & 0xFFFFFFFFFFFFFFFF, _optr(counter), stream_id, _ptr(prob), _ptr(action),
                                       _ptr(log_a), _ptr(task), _stream()), "mtfjsp_enc_select")
    return prob, action, log_a, task


def head_tf32(x, cand, B, rows_per_env, nodes_per_env, in_scale, in_shift, Wa, bias_env, W1, b1, w2, b2, relu=True):
    """mtfjsp_enc_head_tf32: a whole policy head (gather, BatchNorm + ReLU of the producing layer, Linear, per-env bias,
    tanh, Linear, tanh, Linear(128, 1)) in one launch -> scores [B, rows_per_env].  in_scale [G,128]: one affine per
    BatchNorm group of B / G envs (mtfjsp_enc_head_tf32_grouped)."""
    out = torch.empty((B, rows_per_env), dtype=torch.float32, device=x.device)
    if in_scale is not None and in_scale.dim() == 2:
        check(_lib.lib().mtfjsp_enc_head_tf32_grouped(_ptr(x), _optr(cand), B, rows_per_env, nodes_per_env, _ptr(in_scale),
                                                      _ptr(in_shift), 1 if relu else 0, B // in_scale.shape[0], _ptr(Wa),
                                                      _ptr(bias_env), bias_env.shape[0], _ptr(W1), _optr(b1), _ptr(w2), _optr(b2),
                                                      _ptr(out), _stream()), "mtfjsp_enc_head_tf32_grouped")
        return out
    check(_lib.lib().mtfjsp_enc_head_tf32(_ptr(x), _optr(cand), B, rows_per_env, nodes_per_env, _optr(in_scale), _optr(in_shift),
                                          1 if relu else 0, _ptr(Wa), _ptr(bias_env), bias_env.shape[0], _ptr(W1), _optr(b1), _ptr(w2), _optr(b2),
                                          _ptr(out), _stream()), "mtfjsp_enc_head_tf32")
    return out


def gat_trunk_tf32(fea1, fea2, W1p, W2p, Wt, a_src, a_dst, stats=None):
    """mtfjsp_enc_gat_trunk_tf32: input projections + three GAT layers + node-set mean in one launch -> [R,128];
    stats [256] f64 (optional) receives the column sums of the result and of its squares."""
    R = fea1.shape[0]
    out = torch.empty((R, 128), dtype=torch.float32, device=fea1.device)
    check(_lib.lib().mtfjsp_enc_gat_trunk_tf32(_ptr(fea1), _ptr(fea2), _ptr(W1p), _ptr(W2p), _ptr(Wt), _ptr(a_src), _ptr(a_dst),
                                               _ptr(out), _optr(stats), R, _stream()), "mtfjsp_enc_gat_trunk_tf32")
    return out


def gat_trunk_tf32_grouped(fea1, fea2, W1p, W2p, Wt, a_src, a_dst, env_stats, M):
    """mtfjsp_enc_gat_trunk_tf32_grouped: gat_trunk_tf32 over B = R / M envs with env-aligned tiles -> [R,128];
    env_stats [B,1,2,128] f64 receives each env's column sums of the result and of its squares."""
    R = fea1.shape[0]
    out = torch.empty((R, 128), dtype=torch.float32, device=fea1.device)
    check(_lib.lib().mtfjsp_enc_gat_trunk_tf32_grouped(_ptr(fea1), _ptr(fea2), _ptr(W1p), _ptr(W2p), _ptr(Wt), _ptr(a_src),
                                                       _ptr(a_dst), _ptr(out), _ptr(env_stats), R // M, M, _stream()),
          "mtfjsp_enc_gat_trunk_tf32_grouped")
    return out


def _graph_mean_raw(h, in_scale=None, in_shift=None, relu=False):
    B, N, Cc = h.shape
    h = h.contiguous()
    out = torch.empty((B, Cc), dtype=h.dtype, device=h.device)
    if in_scale is not None and in_scale.dim() == 2:  # per-group affine [G,C]
        check(_lib.lib().mtfjsp_enc_graph_mean_grouped(_ptr(h), _ptr(out), B, N, Cc, _ptr(in_scale), _ptr(in_shift), int(relu),
                                                       B // in_scale.shape[0], _stream()), "mtfjsp_enc_graph_mean_grouped")
        return out
    check(_lib.lib().mtfjsp_enc_graph_mean(_ptr(h), _ptr(out), B, N, Cc, _optr(in_scale), _optr(in_shift), int(relu),
                                           _stream()), "mtfjsp_enc_graph_mean")
    return out


def graph_mean(h, in_scale=None, in_shift=None, relu=False):
    if torch.is_grad_enabled() and h.requires_grad:
        if in_scale is not None:
            raise ValueError("the folded input affine is an inference-path option")
        return _GraphMeanFn.apply(h)
    return _graph_mean_raw(h, in_scale, in_shift, relu)


def linear_tf32(x, weight, bias, in_scale=None, in_shift=None, relu=False, stats=None):
    """Z = act(x*in_scale+in_shift) @ weight.T + bias on tcgen05 tensor cores (TF32 operands, FP32 accumulate);
    stats [256] f64 accumulates column sums / sums of squares of Z.  x [rows,K] f32, weight [128,K]."""
    rows, K = x.shape
    assert weight.shape == (128, K) and x.dtype == torch.float32
    z = torch.empty((rows, 128), dtype=torch.float32, device=x.device)
    check(_lib.lib().mtfjsp_enc_linear_tf32(_ptr(x.contiguous()), rows, K, _ptr(weight), _optr(bias), _optr(in_scale),
                                            _optr(in_shift), int(relu), _ptr(z), _optr(stats), _stream()),
          "mtfjsp_enc_linear_tf32")
    return z


def env_stat_pieces(rows_per_env):
    """P of the grouped layers' env_stats [B,P,2,128]: 128-row tile pieces per env."""
    return (rows_per_env + 127) // 128


def linear_tf32_grouped(x, rows_per_env, weight, bias, in_scale, in_shift, relu, env_stats):
    """linear_tf32 over B = rows / rows_per_env envs with env-aligned tiles: in_scale / in_shift [G,128] (one affine per
    group of B / G envs) or None; env_stats [B,P,2,128] f64 receives each env's column sums of Z and Z^2."""
    rows, K = x.shape
    B = rows // rows_per_env
    z = torch.empty((rows, 128), dtype=torch.float32, device=x.device)
    epg = 1 if in_scale is None else B // in_scale.shape[0]
    check(_lib.lib().mtfjsp_enc_linear_tf32_grouped(_ptr(x.contiguous()), B, rows_per_env, K, _ptr(weight), _optr(bias),
                                                    _optr(in_scale), _optr(in_shift), int(relu), epg, _ptr(z), _ptr(env_stats),
                                                    _stream()), "mtfjsp_enc_linear_tf32_grouped")
    return z


def aggregate_linear_tf32_grouped(h, adj_w, adj_src, weight, bias, in_scale, in_shift, relu, env_stats):
    """aggregate_linear_tf32 with [G,128] affines and per-env statistics; None where the form is not available (N > 128)."""
    B, N = h.shape[0], h.shape[1]
    if N > 128:
        return None
    z = torch.empty((B * N, 128), dtype=torch.float32, device=h.device)
    epg = 1 if in_scale is None else B // in_scale.shape[0]
    rc = _lib.lib().mtfjsp_enc_aggregate_linear_tf32_grouped(_ptr(h), B, N, _ptr(adj_w), _ptr(adj_src), _ptr(weight), _optr(bias),
                                                             _optr(in_scale), _optr(in_shift), int(relu), epg, _ptr(z),
                                                             _ptr(env_stats), _stream())
    if rc == -3:  # MTFJSP_E_STATE
        return None
    check(rc, "mtfjsp_enc_aggregate_linear_tf32_grouped")
    return z


def bn_finalize_grouped(env_stats, rows_per_env, groups, gamma, beta, eps=1e-5):
    """env_stats [B,P,2,C] -> scale, shift [groups, C]: BatchNorm with batch statistics per group of B / groups envs."""
    B = env_stats.shape[0]
    Cc = gamma.shape[0]
    scale = torch.empty((groups, Cc), dtype=torch.float32, device=gamma.device)
    shift = torch.empty_like(scale)
    check(_lib.lib().mtfjsp_enc_bn_finalize_grouped(_ptr(env_stats), B, rows_per_env, B // groups, _ptr(gamma), _ptr(beta), eps,
                                                    _ptr(scale), _ptr(shift), Cc, _stream()), "mtfjsp_enc_bn_finalize_grouped")
    return scale, shift


_WGRAD_WS = {}


def wgrad_tf32(gz, x, want_bias=True):
    """Weight / bias gradient of Z = x @ W.T + b on the tcgen05 tensor cores: dW [128,K] = gz.T @ x (TF32 operands,
    FP32 accumulate, partials of the 148 CTAs added in a fixed order), db [128] = column sums of gz."""
    rows, K = x.shape
    assert gz.shape == (rows, 128) and gz.dtype == torch.float32 and x.dtype == torch.float32
    lib = _lib.lib()
    key = (x.device.index, K)
    if key not in _WGRAD_WS:
        _WGRAD_WS[key] = torch.empty(int(lib.mtfjsp_enc_wgrad_workspace_floats(K)), dtype=torch.float32, device=x.device)
    dW = torch.empty((128, K), dtype=torch.float32, device=x.device)
    db = torch.empty(128, dtype=torch.float32, device=x.device) if want_bias else None
    check(lib.mtfjsp_enc_wgrad_tf32(_ptr(gz.contiguous()), _ptr(x.contiguous()), rows, K, _ptr(dW), _optr(db),
                                    _ptr(_WGRAD_WS[key]), _stream()), "mtfjsp_enc_wgrad_tf32")
    return dW, db


def gat_attend(t, a_src, a_dst, mode):
    """Attention + combination (+ELU / node-set mean) of the closed-form 2-node GAT layer, see include/mtfjsp.h."""
    R = t.shape[0] // 2
    out = torch.empty((R if mode == 2 else 2 * R, 128), dtype=torch.float32, device=t.device)
    check(_lib.lib().mtfjsp_enc_gat_attend(_ptr(t), _ptr(a_src), _ptr(a_dst), _ptr(out), R, mode, _stream()),
          "mtfjsp_enc_gat_attend")
    return out


class _GatAttendFn(torch.autograd.Function):
    """gat_attend under autograd for the PPO update: forward = the rollout kernel, backward = one kernel that recomputes
    the attention from t and emits dt plus per-block partial gradients of the two attention vectors."""

    @staticmethod
    def forward(ctx, t, a_src, a_dst, mode):
        t, a_src, a_dst = t.contiguous(), a_src.contiguous(), a_dst.contiguous()
        ctx.save_for_backward(t, a_src, a_dst)
        ctx.mode = mode
        return gat_attend(t, a_src, a_dst, mode)

    @staticmethod
    def backward(ctx, g):
        t, a_src, a_dst = ctx.saved_tensors
        R = t.shape[0] // 2
        lib = _lib.lib()
        nb = int(lib.mtfjsp_enc_gat_attend_bwd_blocks(R))
        dt = torch.empty_like(t)
        parts = torch.empty((nb, 2, 128), dtype=torch.float32, device=t.device)
        check(lib.mtfjsp_enc_gat_attend_bwd(_ptr(t), _ptr(a_src), _ptr(a_dst), _ptr(g.contiguous()), _ptr(dt), _ptr(parts), R,
                                            ctx.mode, _stream()), "mtfjsp_enc_gat_attend_bwd")
        da = parts.sum(dim=0)
        return dt, da[0], da[1], None


def gat_attend_train(t, a_src, a_dst, mode):
    return _GatAttendFn.apply(t, a_src, a_dst, mode)


class _LinearTF32Fn(torch.autograd.Function):
    """nn.Linear (128 outputs) of the PPO re-forward with all three GEMMs on the hand-written tcgen05 kernels:
    forward and input gradient on linear_tf32_kernel (dX = gZ @ W is the same product with W.T as the weight),
    weight / bias gradient on wgrad_tf32_kernel."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x = x.contiguous()
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return linear_tf32(x, weight, bias)

    @staticmethod
    def backward(ctx, gz):
        x, weight = ctx.saved_tensors
        gz = gz.contiguous()
        gx = None
        if ctx.needs_input_grad[0]:
            gx = linear_tf32(gz, weight.t().contiguous(), None) if weight.shape[1] == 128 else gz @ weight
        gw, gb = wgrad_tf32(gz, x, ctx.has_bias)
        return gx, gw, gb


def linear_train(x, weight, bias, tf32):
    """F.linear, or its tcgen05 twin when `tf32` and the shape fits the kernels (128 outputs, K <= 128, K % 4 == 0)."""
    if tf32 and x.is_cuda and weight.shape[0] == 128 and weight.shape[1] <= 128 and weight.shape[1] % 4 == 0 and x.dim() == 2:
        return _LinearTF32Fn.apply(x, weight, bias)
    return F.linear(x, weight, bias)


def bn_finalize(stats, rows, gamma, beta, eps=1e-5):
    Cc = gamma.shape[0]
    scale = torch.empty(Cc, dtype=torch.float32, device=gamma.device)
    shift = torch.empty_like(scale)
    check(_lib.lib().mtfjsp_enc_bn_finalize(_ptr(stats), rows, _ptr(gamma), _ptr(beta), eps, _ptr(scale), _ptr(shift), Cc,
                                            _stream()), "mtfjsp_enc_bn_finalize")
    return scale, shift


def job_actor_keys(hidden=128, in_dim=12):
    """state_dict layout of the reference job actor (read off the shipped tester/IoTJ_MAPPO/*.pth)."""
    H = hidden
    k = {"_input": (H,)}
    for l, din in ((0, in_dim), (1, H)):
        p = "encoder.feature_extract.mlps.%d." % l
        k[p + "linears.0.weight"] = (H, din); k[p + "linears.0.bias"] = (H,)
        for i in (1, 2):
            k[p + "linears.%d.weight" % i] = (H, H); k[p + "linears.%d.bias" % i] = (H,)
        for i in (0, 1):
            for n, s in (("weight", (H,)), ("bias", (H,)), ("running_mean", (H,)), ("running_var", (H,)),
                         ("num_batches_tracked", ())):
                k[p + "batch_norms.%d.%s" % (i, n)] = s
    for name, d in (("encoder.feature_extract.bn.", in_dim), ("encoder.feature_extract.batch_norms.0.", H),
                    ("encoder.feature_extract.batch_norms.1.", H)):
        for n, s in (("weight", (d,)), ("bias", (d,)), ("running_mean", (d,)), ("running_var", (d,)),
                     ("num_batches_tracked", ())):
            k[name + n] = s
    k["o_policy.linears.0.weight"] = (H, 3 * H); k["o_policy.linears.0.bias"] = (H,)
    k["o_policy.linears.1.weight"] = (H, H); k["o_policy.linears.1.bias"] = (H,)
    k["o_policy.linears.2.weight"] = (1, H); k["o_policy.linears.2.bias"] = (1,)
    k["job_critic.linears.0.weight"] = (H, H); k["job_critic.linears.0.bias"] = (H,)
    k["job_critic.linears.1.weight"] = (H, H); k["job_critic.linears.1.bias"] = (H,)
    k["job_critic.linears.2.weight"] = (2, H); k["job_critic.linears.2.bias"] = (2,)
    return k


def machine_actor_keys(hidden=128):
    H = hidden
    k = {}
    for n, s in (("weight", (H,)), ("bias", (H,)), ("running_mean", (H,)), ("running_var", (H,)), ("num_batches_tracked", ())):
        k["bn." + n] = s
    k["m_fea_1_fcl.weight"] = (H, 6); k["m_fea_2_fcl.weight"] = (H, 8)
    k["gat_layer.W"] = (H, H); k["gat_layer.a"] = (1, 2 * H, 1)
    k["fcl_pooling.weight"] = (H, H)
    k["m_policy.linears.0.weight"] = (H, 3 * H); k["m_policy.linears.0.bias"] = (H,)
    k["m_policy.linears.1.weight"] = (H, H); k["m_policy.linears.1.bias"] = (H,)
    k["m_policy.linears.2.weight"] = (1, H); k["m_policy.linears.2.bias"] = (1,)
    k["machine_critic.linears.0.weight"] = (H, H); k["machine_critic.linears.0.bias"] = (H,)
    k["machine_critic.linears.1.weight"] = (H, H); k["machine_critic.linears.1.bias"] = (H,)
    k["machine_critic.linears.2.weight"] = (2, H); k["machine_critic.linears.2.bias"] = (2,)
    return k


def esa_job_actor_keys(hidden=128, in_dim=12):
    """state_dict layout of esa_Operation_Actor_Critic (model/actor_critic.py:945-1205): the job actor with a 4-wide
    critic (read off the shipped tester/ESWA_MPPO/esa_PPO_operation_actor_*.pth)."""
    H = hidden
    k = job_actor_keys(hidden, in_dim)
    k["job_critic.linears.2.weight"] = (4, H); k["job_critic.linears.2.bias"] = (4,)
    return k


def esa_machine_actor_keys(hidden=128):
    """state_dict layout of esa_Machine_Actor (model/actor_critic.py:1207-1404).  `gat_layer.*` and `fcl_pooling.weight`
    are in its state_dict but its forward never reads them."""
    H = hidden
    k = machine_actor_keys(hidden)
    k["m_policy.linears.0.weight"] = (H, 4 * H)
    return k


def seeded_state_dict(keys: dict, seed: int):
    """Deterministic weights for parity fixtures: the same call feeds the reference module (in the build container)
    and this module (on the GPU box), so no checkpoint has to be shipped with the tests."""
    rs = np.random.RandomState(seed)
    sd = {}
    for name, shape in keys.items():
        if name.endswith("num_batches_tracked"):
            sd[name] = torch.tensor(0, dtype=torch.int64)
        elif name.endswith("running_var"):
            sd[name] = torch.ones(shape, dtype=torch.float32)
        elif name.endswith("running_mean"):
            sd[name] = torch.zeros(shape, dtype=torch.float32)
        elif ".batch_norms." in name or name.startswith("bn.") or ".bn." in name:
            v = rs.uniform(0.5, 1.5, size=shape) if name.endswith("weight") else rs.uniform(-0.2, 0.2, size=shape)
            sd[name] = torch.tensor(v, dtype=torch.float32)
        else:
            fan_in = shape[-1] if len(shape) > 1 else max(shape[0], 1)
            if name == "gat_layer.a":
                fan_in = shape[1]
            sd[name] = torch.tensor(rs.standard_normal(size=shape) / np.sqrt(fan_in), dtype=torch.float32)
    return sd


def bn_forward(x, w, b, eps, groups, relu):
    """Grouped BatchNorm1d with batch statistics (+ReLU) on the device: -> y, mean [G,C], rstd [G,C]."""
    Cc = x.shape[-1]
    x = x.contiguous()
    R = x.numel() // (groups * Cc)
    y = torch.empty_like(x)
    mean = torch.empty((groups, Cc), dtype=torch.float32, device=x.device)
    rstd = torch.empty_like(mean)
    ws = torch.empty((groups, 2, Cc), dtype=torch.float64, device=x.device)
    check(_lib.lib().mtfjsp_enc_bn_fwd(_ptr(x), _ptr(w.contiguous()), _ptr(b.contiguous()), float(eps), groups, R, Cc, int(relu),
                                       _ptr(y), _ptr(mean), _ptr(rstd), _ptr(ws), _stream()), "mtfjsp_enc_bn_fwd")
    return y, mean, rstd


def bn_backward(x, gy, w, b, mean, rstd, groups, relu):
    """-> dx, dgamma [C], dbeta [C]."""
    Cc = x.shape[-1]
    R = x.numel() // (groups * Cc)
    gy = gy.contiguous()
    dx = torch.empty_like(x)
    sums = torch.empty((groups, 2, Cc), dtype=torch.float64, device=x.device)
    check(_lib.lib().mtfjsp_enc_bn_bwd(_ptr(x), _ptr(gy), _ptr(w.contiguous()), _ptr(b.contiguous()), _ptr(mean), _ptr(rstd),
                                       groups, R, Cc, int(relu), _ptr(dx), _ptr(sums), _stream()), "mtfjsp_enc_bn_bwd")
    tot = sums.sum(dim=0)
    return dx, tot[1].float(), tot[0].float()


class _GroupBNFn(torch.autograd.Function):
    """BatchNorm1d with batch statistics per row group (+ optional ReLU) that keeps only its input for the backward:
    the PPO re-forward holds ~20 of these per network, so the usual elementwise chain (centred, scaled, shifted,
    rectified copies) would be most of the activation memory.  Kernels: csrc/mtfjsp_encoder.cu bn_*_kernel."""

    @staticmethod
    def forward(ctx, x, w, b, eps, groups, relu):
        x = x.contiguous()
        y, mean, rstd = bn_forward(x, w, b, eps, groups, relu)
        ctx.save_for_backward(x, w, b, mean, rstd)
        ctx.groups, ctx.relu = groups, relu
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w, b, mean, rstd = ctx.saved_tensors
        dx, dgamma, dbeta = bn_backward(x, gy, w, b, mean, rstd, ctx.groups, ctx.relu)
        return dx, dgamma, dbeta, None, None, None


def _bn_train(x, w, b, eps=1e-5, groups=1, relu=False):
    """BatchNorm1d with batch statistics (the reference never leaves train mode), optionally followed by ReLU.
    groups > 1: the rows are `groups` consecutive blocks, each normalised with its own statistics -- one block per
    buffered step, so a batched PPO re-forward sees exactly the statistics of the reference's one-step-at-a-time loop
    (ppo_algorithm.py:739-775)."""
    if torch.is_grad_enabled() and (x.requires_grad or w.requires_grad):
        return _GroupBNFn.apply(x, w, b, eps, groups, relu)
    if groups == 1:
        y = F.batch_norm(x, None, None, w, b, True, 0.0, eps)
        return F.relu(y) if relu else y
    return bn_forward(x, w, b, eps, groups, relu)[0]


class _Params:
    def __init__(self, keys, state_dict, device, trainable=False):
        missing = [k for k in keys if k not in state_dict]
        extra = [k for k in state_dict if k not in keys]
        if missing or extra:
            raise KeyError("state_dict mismatch: missing %s unexpected %s" % (missing, extra))
        self.p = {}
        for k, shape in keys.items():
            t = torch.as_tensor(state_dict[k])
            if tuple(t.shape) != tuple(shape):
                raise ValueError("%s: shape %s, expected %s" % (k, tuple(t.shape), tuple(shape)))
            self.p[k] = t.to(device=device, dtype=torch.float32 if t.is_floating_point() else t.dtype).contiguous().clone()
            if trainable and self.is_parameter(k):
                self.p[k].requires_grad_(True)

    @staticmethod
    def is_parameter(k):
        return not k.endswith(("running_mean", "running_var", "num_batches_tracked"))

    def __getitem__(self, k):
        return self.p[k]

    def detached(self):
        """Same storage, no autograd: the view an inference twin reads while the optimiser updates in place."""
        v = object.__new__(_Params)
        v.p = {k: t.detach() for k, t in self.p.items()}
        return v

    def parameters(self):
        """Learnable tensors in state_dict order (what `module.parameters()` yields in the reference)."""
        return [t for k, t in self.p.items() if self.is_parameter(k)]

    def state_dict(self):
        return {k: t.detach().clone() for k, t in self.p.items()}


def _mlp3_tanh_tf32(w, prefix, x):
    """_mlp3_tanh with the two 128 -> 128 layers on the tcgen05 kernel (rollout path, value heads on pooled [B,128])."""
    h = torch.tanh(linear_tf32(x.contiguous(), w[prefix + "linears.0.weight"], w[prefix + "linears.0.bias"]))
    h = torch.tanh(linear_tf32(h, w[prefix + "linears.1.weight"], w[prefix + "linears.1.bias"]))
    return F.linear(h, w[prefix + "linears.2.weight"], w[prefix + "linears.2.bias"])


def _mlp3_tanh(w, prefix, x):
    """MLPActor / MLPCritic with three linears and tanh between them (model/gcn_mlp.py:258-320)."""
    h = torch.tanh(F.linear(x, w[prefix + "linears.0.weight"], w[prefix + "linears.0.bias"]))
    h = torch.tanh(F.linear(h, w[prefix + "linears.1.weight"], w[prefix + "linears.1.bias"]))
    return F.linear(h, w[prefix + "linears.2.weight"], w[prefix + "linears.2.bias"])


class _GraphEncoder:
    """GraphCNN (model/gcn_mlp.py:109-197) over the env's ELL adjacency; shared by the job actor and the global critic."""

    def _mlp(self, l, x, groups=1):  # gcn_mlp.py:238-249
        w = self.w
        p = "encoder.feature_extract.mlps.%d." % l
        h = x
        tf32 = getattr(self, "train_tf32", False)  # PPOConfig.encoder_tf32: the update's encoder GEMMs on tcgen05
        for i in (0, 1):
            h = linear_train(h, w[p + "linears.%d.weight" % i], w[p + "linears.%d.bias" % i], tf32)
            h = _bn_train(h, w[p + "batch_norms.%d.weight" % i], w[p + "batch_norms.%d.bias" % i], groups=groups, relu=True)
        return linear_train(h, w[p + "linears.2.weight"], w[p + "linears.2.bias"], tf32)

    def encode(self, task_fea, adj_w, adj_src, groups=1, adj_dst=None):
        """GraphCNN.forward (gcn_mlp.py:160-197): two rounds of aggregate -> MLP -> BN -> ReLU, then mean pooling.
        task_fea [B,N,12] f32, adj_w [B,N,2] f32, adj_src [B,N] i16 -> (pooled [B,H], nodes [B,N,H]).
        groups: B is `groups` consecutive env batches with separate BatchNorm statistics (see _bn_train)."""
        B = task_fea.shape[0]
        w = self.w
        h = task_fea.to(torch.float32)
        if self.precision == "tf32":
            if groups != 1:
                return self._encode_tf32_grouped(h, adj_w, adj_src, groups)
            return self._encode_tf32(h, adj_w, adj_src)
        for l in (0, 1):
            pooled = aggregate(h, adj_w, adj_src, adj_dst=adj_dst)                  # gcn_mlp.py:125-149
            z = self._mlp(l, pooled.reshape(B * self.N, -1), groups)
            z = _bn_train(z, w["encoder.feature_extract.batch_norms.%d.weight" % l],
                          w["encoder.feature_extract.batch_norms.%d.bias" % l], groups=groups, relu=True)   # gcn_mlp.py:154-157
            h = z.reshape(B, self.N, self.H)
        self._pending = None
        return graph_mean(h), h                                                    # gcn_mlp.py:192

    def _encode_tf32(self, h, adj_w, adj_src):
        """Same network on the fused tensor-core layer: every activation is written once and read once; the
        BatchNorm of a layer is applied by its consumer (next layer's prologue, next aggregation, pooling)."""
        w = self.w
        B = h.shape[0]
        rows = B * self.N
        sc = sh = None
        for l in (0, 1):
            p = "encoder.feature_extract.mlps.%d." % l
            z = isc = ish = None
            for i in (0, 1, 2):
                stats = torch.zeros(256, dtype=torch.float64, device=h.device)
                if i == 0:  # aggregation + first layer: one launch where the size allows it
                    if l > 0:
                        z = aggregate_linear_tf32(h, adj_w, adj_src, w[p + "linears.0.weight"], w[p + "linears.0.bias"], sc, sh,
                                                  relu=True, stats=stats)
                    if z is None:
                        pooled = aggregate(h, adj_w, adj_src, sc, sh, relu=sc is not None).reshape(rows, -1)
                        z = linear_tf32(pooled, w[p + "linears.0.weight"], w[p + "linears.0.bias"], None, None, stats=stats)
                else:
                    z = linear_tf32(z, w[p + "linears.%d.weight" % i], w[p + "linears.%d.bias" % i], isc, ish,
                                    relu=isc is not None, stats=stats)
                if i < 2:
                    isc, ish = bn_finalize(stats, rows, w[p + "batch_norms.%d.weight" % i], w[p + "batch_norms.%d.bias" % i])
                else:
                    sc, sh = bn_finalize(stats, rows, w["encoder.feature_extract.batch_norms.%d.weight" % l],
                                         w["encoder.feature_extract.batch_norms.%d.bias" % l])
            h = z.reshape(B, self.N, self.H)
        self._pending = (sc, sh)  # outer BatchNorm + ReLU of the last layer, applied by the consumers below
        return graph_mean(h, sc, sh, relu=True), h

    def _encode_tf32_grouped(self, h, adj_w, adj_src, groups):
        """_encode_tf32 with a BatchNorm group per B / groups consecutive envs: the grouped kernels write per-env
        statistics (summed in a fixed env-local order, so an env's results do not depend on its batch position) and every
        consumer applies the [groups, 128] affine of its env's group."""
        w = self.w
        B, N = h.shape[0], self.N
        if B % groups:
            raise ValueError("groups must divide the batch")
        rows = B * N
        env_stats = torch.empty((B, env_stat_pieces(N), 2, 128), dtype=torch.float64, device=h.device)
        fin = lambda name: bn_finalize_grouped(env_stats, N, groups, w[name + "weight"], w[name + "bias"])
        adj_w, adj_src = adj_w.contiguous(), adj_src.contiguous()
        sc = sh = None
        for l in (0, 1):
            p = "encoder.feature_extract.mlps.%d." % l
            z = None
            if l > 0:
                z = aggregate_linear_tf32_grouped(h, adj_w, adj_src, w[p + "linears.0.weight"], w[p + "linears.0.bias"], sc, sh,
                                                  True, env_stats)
            if z is None:
                pooled = aggregate(h, adj_w, adj_src, sc, sh, relu=sc is not None).reshape(rows, -1)
                z = linear_tf32_grouped(pooled, N, w[p + "linears.0.weight"], w[p + "linears.0.bias"], None, None, False, env_stats)
            isc, ish = fin(p + "batch_norms.0.")
            z = linear_tf32_grouped(z, N, w[p + "linears.1.weight"], w[p + "linears.1.bias"], isc, ish, True, env_stats)
            isc, ish = fin(p + "batch_norms.1.")
            z = linear_tf32_grouped(z, N, w[p + "linears.2.weight"], w[p + "linears.2.bias"], isc, ish, True, env_stats)
            sc, sh = fin("encoder.feature_extract.batch_norms.%d." % l)
            h = z.reshape(B, N, self.H)
        self._pending = (sc, sh)  # [groups, 128]
        return graph_mean(h, sc, sh, relu=True), h

    def candidate_features(self, nodes, candidate):
        cf = torch.gather(nodes, 1, candidate.long().unsqueeze(-1).expand(-1, self.J, self.H))   # actor_critic.py:197-207
        if self._pending is not None:
            sc, sh = self._pending
            if sc.dim() == 2:  # [G,128]: the affine of each env's BatchNorm group
                epg = cf.shape[0] // sc.shape[0]
                sc, sh = sc.repeat_interleave(epg, 0).unsqueeze(1), sh.repeat_interleave(epg, 0).unsqueeze(1)
            cf = torch.relu(cf * sc + sh)
        return cf

    def parameters(self):
        return self.w.parameters()

    def state_dict(self):
        return self.w.state_dict()


class _Twin:
    def inference_twin(self, precision="tf32"):
        """A second handle on the SAME weights for rollouts (no autograd, optionally the tcgen05 path) while this
        object trains them; call `refresh()` on the twin after optimiser steps (re-derives cached layouts in place,
        so captured CUDA graphs stay valid)."""
        _check_precision(precision, self.H)
        t = object.__new__(type(self))
        t.__dict__.update(self.__dict__)
        t.__dict__.pop("_twins", None)
        t.w = self.w.detached()
        t.precision = precision
        t._pending = None
        t._dcache = {}
        self.__dict__.setdefault("_twins", []).append(weakref.ref(t))  # MAPPOUpdate.update refreshes them
        return t

    def refresh_twins(self):
        """Re-derives the cached weight layouts of every live inference twin of this network (after optimiser steps)."""
        alive = []
        for r in self.__dict__.get("_twins", []):
            t = r()
            if t is not None:
                t.refresh()
                alive.append(r)
        if "_twins" in self.__dict__:
            self._twins = alive

    def _derived(self, name, fn):
        """Weight layouts derived for the tensor-core path (transposes, column blocks), built once per object."""
        c = self.__dict__.setdefault("_dcache", {})
        if name not in c:
            c[name] = (fn().contiguous(), fn)
        return c[name][0]

    def refresh(self):
        for t, fn in self.__dict__.get("_dcache", {}).values():
            t.copy_(fn())

    def _head_tf32(self, prefix, per_row, env_terms, rows_per_env, in_scale=None, in_shift=None, cand=None, relu=True):
        """First two layers of a 3-layer tanh MLP whose input is cat(per_row [B*r,H], env_term_0 [B,H], env_term_1 [B,H]):
        the per-env blocks of the first weight matrix are applied once per env and added as a bias, the per-row block
        and the second layer run on the tcgen05 kernel -- no [B*r, 3H] concatenation, a third of the GEMM work."""
        w, H = self.w, self.H
        W0 = w[prefix + "linears.0.weight"]
        Wa = self._derived(prefix + "W0a", lambda: W0[:, :H])
        bias = w[prefix + "linears.0.bias"]
        for k, e in enumerate(env_terms):
            Wk = self._derived(prefix + "W0%d" % (k + 1), lambda k=k: W0[:, (k + 1) * H:(k + 2) * H])
            term = linear_tf32(e.contiguous(), Wk, bias if k == 0 else None)  # the layer's own bias rides on the first term
            bias = term if k == 0 else bias + term
        bias = (bias if bias.dim() == 2 else bias.unsqueeze(0)).contiguous()
        w2 = self._derived(prefix + "w2", lambda: w[prefix + "linears.2.weight"].reshape(-1))
        if cand is not None:  # per_row = the node embeddings [B, nodes, H]; the kernel gathers the candidate rows itself
            B, nodes = per_row.shape[0], per_row.shape[1]
        else:
            B, nodes = per_row.shape[0] // rows_per_env, 0
        return head_tf32(per_row, cand, B, rows_per_env, nodes, in_scale, in_shift, Wa, bias,
                         w[prefix + "linears.1.weight"], w[prefix + "linears.1.bias"], w2, w[prefix + "linears.2.bias"], relu=relu)


def _head_train(self, prefix, per_row, env_terms, rows_per_env):
    """Training-path twin of _Twin._head_tf32 (PPOConfig.encoder_tf32): the same decomposition of the first layer of a
    3-layer tanh MLP over cat(per_row, env_term_0, env_term_1) -- per-env column blocks applied once per env instead of
    once per row -- with the two [rows,128] x [128,128] products on the tcgen05 kernels under autograd (linear_train)."""
    w, H = self.w, self.H
    W0 = w[prefix + "linears.0.weight"]
    z = linear_train(per_row, W0[:, :H].contiguous(), None, True)
    bias = w[prefix + "linears.0.bias"]
    for k, e in enumerate(env_terms):
        bias = bias + F.linear(e, W0[:, (k + 1) * H:(k + 2) * H])
    B = per_row.shape[0] // rows_per_env
    z = torch.tanh(z.view(B, rows_per_env, H) + (bias.unsqueeze(1) if bias.dim() == 2 else bias)).view(-1, H)
    z = torch.tanh(linear_train(z, w[prefix + "linears.1.weight"], w[prefix + "linears.1.bias"], True))
    return F.linear(z, w[prefix + "linears.2.weight"], w[prefix + "linears.2.bias"]).view(B, rows_per_env)


def _check_precision(precision, hidden):
    if precision not in ("fp32", "tf32"):
        raise ValueError("precision must be 'fp32' or 'tf32'")
    if precision == "tf32" and hidden != 128:
        raise ValueError("the tcgen05 layer kernel is built for hidden = 128")


class JobActor(_GraphEncoder, _Twin):
    """Forward of Operation_Actor_JointAction_selfCritic (model/actor_critic.py:104-296) on native observations."""

    n_values = 2  # width of job_v
    _keys = staticmethod(job_actor_keys)

    def __init__(self, state_dict, n_job, n_machine, hidden=128, in_dim=12, device=None, precision="fp32", trainable=False):
        """precision "fp32": library FP32 GEMMs, bit-for-bit the reference's arithmetic types;
        "tf32": the fused tcgen05 layer kernel (hidden must be 128) -- BatchNorm folded into prologue/epilogue."""
        self.J, self.M, self.N, self.H = n_job, n_machine, n_job * n_machine, hidden
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.w = _Params(self._keys(hidden, in_dim), state_dict, self.device, trainable)
        _check_precision(precision, hidden)
        self.precision = precision
        self._pending = None

    def evaluate(self, task_fea, adj_w, adj_src, candidate, h_g_m_pooled, mask_operation, groups=1, adj_dst=None,
                 return_logits=False):
        """Action distribution and local values without sampling: prob [B,J], h_g_o_pooled [B,H], job_v [B,2].
        h_g_m_pooled [B,H] or None (the learned `_input` vector stands in, actor_critic.py:232-240).
        return_logits: the unmasked scores instead of prob (the rollout's one-launch selection masks them itself)."""
        w = self.w
        pooled, nodes = self.encode(task_fea, adj_w, adj_src, groups, adj_dst)
        if self.precision == "tf32":
            sc, sh = self._pending
            gmv = w["_input"].unsqueeze(0) if h_g_m_pooled is None else h_g_m_pooled
            s = self._head_tf32("o_policy.", nodes, (pooled, gmv), self.J, sc, sh, cand=candidate.to(torch.int32).contiguous())
        elif getattr(self, "train_tf32", False):
            cf = self.candidate_features(nodes, candidate)
            gmv = w["_input"].unsqueeze(0) if h_g_m_pooled is None else h_g_m_pooled
            s = _head_train(self, "o_policy.", cf.reshape(-1, self.H), (pooled, gmv), self.J)
        else:
            cf = self.candidate_features(nodes, candidate)
            gm = w["_input"][None, None, :].expand_as(cf) if h_g_m_pooled is None else h_g_m_pooled.unsqueeze(-2).expand_as(cf)
            x = torch.cat((cf, pooled.unsqueeze(-2).expand_as(cf), gm), dim=-1)          # actor_critic.py:244-247
            s = _mlp3_tanh(w, "o_policy.", x).squeeze(-1)
        job_v = (_mlp3_tanh_tf32 if self.precision == "tf32" else _mlp3_tanh)(w, "job_critic.", pooled)
        if return_logits:
            return s, pooled, job_v
        s = s.masked_fill(mask_operation.bool(), float("-inf"))                          # actor_critic.py:266-268
        prob = F.softmax(s, dim=-1)
        return prob, pooled, job_v

    def forward(self, task_fea, adj_w, adj_src, candidate, h_g_m_pooled, mask_operation, greedy=False, generator=None, rng=None,
                groups=1):
        """-> task_index [B], action_index [B] (job), log_a [B], prob [B,J], h_g_o_pooled [B,H], job_v [B,2].
        rng = (seed, device step counter): sampling by the one-launch selection kernel (`select`) instead of
        torch.multinomial on `generator`.  groups: BatchNorm groups of B / groups consecutive envs (see `encode`)."""
        if rng is not None and not greedy:
            s, pooled, job_v = self.evaluate(task_fea, adj_w, adj_src, candidate, h_g_m_pooled, mask_operation, groups=groups,
                                             return_logits=True)
            prob, a, log_a, task_index = select(s, mask_operation, candidate.to(torch.int32).contiguous(), 1.0, False, rng, 0)
            return task_index, a, log_a, prob, pooled, job_v
        prob, pooled, job_v = self.evaluate(task_fea, adj_w, adj_src, candidate, h_g_m_pooled, mask_operation, groups=groups)
        if greedy:                                                                       # agent_func.py greedy / sample
            a = prob.argmax(dim=-1)
        else:
            a = torch.multinomial(prob, 1, generator=generator).squeeze(-1)
        log_a = torch.log(prob.gather(1, a.unsqueeze(-1)).squeeze(-1))
        task_index = candidate.long().gather(1, a.unsqueeze(-1)).squeeze(-1)
        return task_index, a, log_a, prob, pooled, job_v


class _MachineTrunk:
    """Machine-node embedding shared by the machine actor and the global critic (actor_critic.py:381-440, 666-700):
    two input projections, the GAT layer (model/gat.py:68-159) applied three times on the fixed 2-node graph
    [[1,1],[0,1]] in closed form, BatchNorm, mean over machines."""

    def _gat(self, h1, h2):
        """GATLayer.forward (gat.py:82-159): node 1 attends to {1, 2}, node 2 to itself."""
        W, a = self.w["gat_layer.W"], self.w["gat_layer.a"]
        H = self.H
        if getattr(self, "train_tf32", False):  # the PPO update: same product under autograd (linear_train)
            t = linear_train(torch.cat((h1, h2), dim=0), W.t().contiguous(), None, True)
            t1, t2 = t[: h1.shape[0]], t[h1.shape[0]:]
        else:
            t1, t2 = h1 @ W, h2 @ W
        a_src, a_dst = a[0, :H, 0], a[0, H:, 0]
        e11 = F.leaky_relu(t1 @ a_src + t1 @ a_dst, 0.2)
        e12 = F.leaky_relu(t1 @ a_src + t2 @ a_dst, 0.2)
        att = torch.softmax(torch.stack((e11, e12), dim=-1), dim=-1)
        return att[..., 0:1] * t1 + att[..., 1:2] * t2, t2

    def trunk(self, machine_fea_1, machine_fea_2, groups=1):
        """machine_fea_1 [B,M,6], machine_fea_2 [B,M,8] -> (nodes [B,M,H], pooled [B,H])."""
        w = self.w
        B = machine_fea_1.shape[0]
        if self.precision == "tf32":
            return self._trunk_tf32(machine_fea_1, machine_fea_2, groups)
        if getattr(self, "train_tf32", False) and self.H == 128 and machine_fea_1.is_cuda:
            return self._trunk_train_fused(machine_fea_1, machine_fea_2, groups)
        h1 = F.linear(machine_fea_1.to(torch.float32), w["m_fea_1_fcl.weight"]).reshape(B * self.M, self.H)
        h2 = F.linear(machine_fea_2.to(torch.float32), w["m_fea_2_fcl.weight"]).reshape(B * self.M, self.H)
        h1, h2 = self._gat(h1, h2)
        h1, h2 = self._gat(F.elu(h1), F.elu(h2))
        h1, h2 = self._gat(F.elu(h1), F.elu(h2))
        hm = torch.stack((h1, h2), dim=1).mean(dim=-2)                                   # actor_critic.py:420
        nodes = _bn_train(hm, w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, self.M, self.H)   # actor_critic.py:434
        return nodes, nodes.mean(dim=1)

    def _trunk_train_fused(self, machine_fea_1, machine_fea_2, groups):
        """PPO-update twin of _trunk_tf32 (PPOConfig.encoder_tf32): per GAT layer one tcgen05 projection of both node sets
        and one attention / combination / ELU kernel, each with a hand-written backward, instead of ~20 library
        elementwise launches forward and as many backward per layer."""
        w, H = self.w, self.H
        B = machine_fea_1.shape[0]
        R = B * self.M
        h1 = F.linear(machine_fea_1.to(torch.float32).reshape(R, 6), w["m_fea_1_fcl.weight"])
        h2 = F.linear(machine_fea_2.to(torch.float32).reshape(R, 8), w["m_fea_2_fcl.weight"])
        buf = torch.cat((h1, h2), dim=0)
        Wt = w["gat_layer.W"].t().contiguous()
        a = w["gat_layer.a"]
        a_src, a_dst = a[0, :H, 0], a[0, H:, 0]
        for layer in range(3):
            t = linear_train(buf, Wt, None, True)
            buf = gat_attend_train(t, a_src, a_dst, 1 if layer < 2 else 2)
        nodes = _bn_train(buf, w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, self.M, H)
        return nodes, nodes.mean(dim=1)

    def _trunk_tf32(self, machine_fea_1, machine_fea_2, groups):
        """Rollout path: input projections, three GAT layers and the node-set mean in one tcgen05 launch
        (gat_trunk_tf32); one BatchNorm group, groups of several envs, or one env per group."""
        w, H = self.w, self.H
        B = machine_fea_1.shape[0]
        R = B * self.M
        f1 = machine_fea_1.to(torch.float32).reshape(R, 6).contiguous()
        f2 = machine_fea_2.to(torch.float32).reshape(R, 8).contiguous()
        Wt = self._derived("gat_Wt", lambda: self.w["gat_layer.W"].t())
        a_src = self._derived("gat_a_src", lambda: self.w["gat_layer.a"][0, :H, 0])
        a_dst = self._derived("gat_a_dst", lambda: self.w["gat_layer.a"][0, H:, 0])
        self._pending_m = None
        if groups == 1:
            # the trunk kernel leaves the BatchNorm statistics behind; the normalisation itself is applied by the consumers
            # (the policy head's prologue; the mean over machines commutes with the per-column affine)
            stats = torch.zeros(256, dtype=torch.float64, device=f1.device)
            buf = gat_trunk_tf32(f1, f2, w["m_fea_1_fcl.weight"], w["m_fea_2_fcl.weight"], Wt, a_src, a_dst, stats)
            sc, sh = bn_finalize(stats, R, w["bn.weight"], w["bn.bias"])
            self._pending_m = (sc, sh)
            return buf.view(B, self.M, H), _graph_mean_raw(buf.view(B, self.M, H), sc, sh, relu=False)
        if B > groups:
            # groups of several envs (training rollouts, Rollout(bn_group_envs=...)): per-env statistics from the trunk
            # kernel; groups of one env (per-instance validation) keep the separate BatchNorm pass below, whose decisions
            # tests/test_grouped_bn.py pins bit for bit against one-instance batches
            return self._trunk_tf32_grouped(f1, f2, Wt, a_src, a_dst, groups)
        buf = gat_trunk_tf32(f1, f2, w["m_fea_1_fcl.weight"], w["m_fea_2_fcl.weight"], Wt, a_src, a_dst)
        nodes = _bn_train(buf, w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, self.M, H)
        return nodes, nodes.mean(dim=1)

    def _trunk_tf32_grouped(self, f1, f2, Wt, a_src, a_dst, groups):
        """_trunk_tf32 with a BatchNorm group per B / groups envs: per-env statistics from the grouped trunk kernel (an
        env's are the same bits at any batch position), the [groups, 128] affines applied by the pooling and the policy
        head's prologue.  f1 [B*M,6], f2 [B*M,8] f32."""
        w, H = self.w, self.H
        B = f1.shape[0] // self.M
        if B % groups:
            raise ValueError("groups must divide the batch")
        env_stats = torch.empty((B, 1, 2, 128), dtype=torch.float64, device=f1.device)
        buf = gat_trunk_tf32_grouped(f1, f2, w["m_fea_1_fcl.weight"], w["m_fea_2_fcl.weight"], Wt, a_src, a_dst, env_stats, self.M)
        sc, sh = bn_finalize_grouped(env_stats, self.M, groups, w["bn.weight"], w["bn.bias"])
        self._pending_m = (sc, sh)
        return buf.view(B, self.M, H), _graph_mean_raw(buf.view(B, self.M, H), sc, sh, relu=False)

    def parameters(self):
        return self.w.parameters()

    def state_dict(self):
        return self.w.state_dict()


class MachineActor(_MachineTrunk, _Twin):
    """Forward of Machine_Actor_JointAction_selfGAT_selfCritic (model/actor_critic.py:359-498).  With 1 < groups < B the
    tf32 path takes per-env statistics from the grouped trunk kernel and applies the [groups, 128] affines in the pooling
    and the policy head.  With one env per group it normalises through mtfjsp_enc_bn_fwd, which takes at most 65,535
    groups per call (its grid.y)."""

    n_values = 2  # width of machine_v

    def __init__(self, state_dict, n_machine, hidden=128, device=None, precision="fp32", trainable=False):
        self.M, self.H = n_machine, hidden
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.w = _Params(machine_actor_keys(hidden), state_dict, self.device, trainable)
        _check_precision(precision, hidden)
        self.precision = precision

    def heads(self, nodes, pooled, h_pooled_o, machine_mask, return_logits=False):
        w = self.w
        B = nodes.shape[0]
        if self.precision == "tf32":
            sc, sh = self.__dict__.get("_pending_m") or (None, None)  # BatchNorm left to this consumer by _trunk_tf32
            s = self._head_tf32("m_policy.", nodes.reshape(-1, self.H), (pooled, h_pooled_o), self.M, sc, sh, relu=False) * 10
        elif getattr(self, "train_tf32", False):
            s = _head_train(self, "m_policy.", nodes.reshape(-1, self.H), (pooled, h_pooled_o), self.M) * 10
        else:
            x = torch.cat((nodes, pooled.unsqueeze(1).expand_as(nodes), h_pooled_o.unsqueeze(1).expand_as(nodes)), dim=-1)
            s = _mlp3_tanh(w, "m_policy.", x).squeeze(-1) * 10
        machine_v = (_mlp3_tanh_tf32 if self.precision == "tf32" else _mlp3_tanh)(w, "machine_critic.", pooled)
        if return_logits:
            return s, machine_v
        s = s.masked_fill(machine_mask.reshape(B, self.M).bool(), float("-inf"))
        return F.softmax(s, dim=-1), machine_v

    def forward(self, machine_fea_1, machine_fea_2, h_pooled_o, machine_mask, groups=1, return_logits=False):
        """machine_fea_1 [B,M,6], machine_fea_2 [B,M,8] f32, h_pooled_o [B,H], machine_mask [B,M] (1 = infeasible)
        -> mch_prob [B,M], h_pooled [B,H], machine_v [B,2]."""
        nodes, pooled = self.trunk(machine_fea_1, machine_fea_2, groups)
        prob, machine_v = self.heads(nodes, pooled, h_pooled_o, machine_mask, return_logits)
        return prob, pooled, machine_v


class EsaJobActor(JobActor):
    """Forward of esa_Operation_Actor_Critic (model/actor_critic.py:945-1205), the ESA-PPO baseline's job actor: the
    JobActor network with a 4-wide job critic.  Inference only (the reference has no ESA training)."""

    n_values = 4
    _keys = staticmethod(esa_job_actor_keys)

    def __init__(self, state_dict, n_job, n_machine, hidden=128, in_dim=12, device=None, precision="fp32"):
        super().__init__(state_dict, n_job, n_machine, hidden, in_dim, device, precision)


_ESA_WS = {}


class EsaMachineActor(_Twin):
    """Forward of esa_Machine_Actor (model/actor_critic.py:1207-1404), the ESA-PPO baseline's machine actor.  No GAT:
        h1 = BN(fea1 W1^T), h2 = BN(fea2 W2^T)    (one BatchNorm module, batch statistics of each call)
        pooled = (mean_m h1 + mean_m h2) / 2,   scores = 10 m_policy(cat(h1, h2, pooled, h_pooled_o)),
        machine_v = machine_critic(pooled)
    precision "fp32": that chain literally on library FP32 GEMMs (per-instance BatchNorm groups work);
    "tf32": BatchNorm and both projections folded into the first m_policy layer (K = 14 on the raw features), the
    statistics from the feature moments -- mtfjsp_enc_esa_mach_stats + mtfjsp_enc_esa_mach_fold + mtfjsp_enc_esa_mach_head_tf32,
    no [B*M,128] intermediate; one BatchNorm group."""

    n_values = 2

    def __init__(self, state_dict, n_machine, hidden=128, device=None, precision="fp32"):
        self.M, self.H = n_machine, hidden
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.w = _Params(esa_machine_actor_keys(hidden), state_dict, self.device)
        _check_precision(precision, hidden)
        self.precision = precision

    def forward(self, machine_fea_1, machine_fea_2, h_pooled_o, machine_mask, groups=1, return_logits=False):
        """machine_fea_1 [B,M,6], machine_fea_2 [B,M,8], h_pooled_o [B,H], machine_mask [B,M] (1 = infeasible)
        -> mch_prob [B,M] (the x10 scores with return_logits), h_pooled [B,H], machine_v [B,2]."""
        w = self.w
        B = machine_fea_1.shape[0]
        f1 = machine_fea_1.to(torch.float32).reshape(B * self.M, 6).contiguous()
        f2 = machine_fea_2.to(torch.float32).reshape(B * self.M, 8).contiguous()
        if self.precision == "tf32":
            if groups != 1:
                raise ValueError("the tf32 ESA machine actor is the rollout path: one BatchNorm group")
            s, pooled = self._scores_fused(f1, f2, h_pooled_o.contiguous(), B)
            machine_v = _mlp3_tanh_tf32(w, "machine_critic.", pooled)
        else:
            s, pooled = self._scores_fp32(f1, f2, h_pooled_o, B, groups)
            machine_v = _mlp3_tanh(w, "machine_critic.", pooled)
        if return_logits:
            return s, pooled, machine_v
        s = s.masked_fill(machine_mask.reshape(B, self.M).bool(), float("-inf"))     # actor_critic.py:1383-1388
        return F.softmax(s, dim=-1), pooled, machine_v

    def _scores_fp32(self, f1, f2, h_pooled_o, B, groups):
        w, M, H = self.w, self.M, self.H
        h1 = _bn_train(F.linear(f1, w["m_fea_1_fcl.weight"]), w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, M, H)
        h2 = _bn_train(F.linear(f2, w["m_fea_2_fcl.weight"]), w["bn.weight"], w["bn.bias"], groups=groups).reshape(B, M, H)
        pooled = (h1.mean(dim=1) + h2.mean(dim=1)) / 2                                  # actor_critic.py:1354-1356
        x = torch.cat((h1, h2, pooled.unsqueeze(1).expand_as(h1), h_pooled_o.unsqueeze(1).expand_as(h1)), dim=-1)
        return _mlp3_tanh(w, "m_policy.", x).squeeze(-1) * 10, pooled

    def _env_bias(self, pooled, h_pooled_o, b0):
        """b0 + W0c pooled + W0d h_pooled_o [B,128]: the per-env column blocks of the first m_policy layer."""
        w, H = self.w, self.H
        W0 = w["m_policy.linears.0.weight"]
        Wc = self._derived("esa_W0c", lambda: W0[:, 2 * H:3 * H])
        Wd = self._derived("esa_W0d", lambda: W0[:, 3 * H:])
        return linear_tf32(pooled, Wc, b0) + linear_tf32(h_pooled_o, Wd, None)

    def _scores_fused(self, f1, f2, h_pooled_o, B):
        w, M = self.w, self.M
        lib = _lib.lib()
        dev = f1.device
        if dev.index not in _ESA_WS:
            _ESA_WS[dev.index] = torch.empty(int(lib.mtfjsp_enc_esa_mach_stats_workspace_doubles()), dtype=torch.float64, device=dev)
        moments = torch.empty(114, dtype=torch.float64, device=dev)
        env_mean = torch.empty((B, 16), dtype=torch.float32, device=dev)
        check(lib.mtfjsp_enc_esa_mach_stats(_ptr(f1), _ptr(f2), B, M, _ptr(moments), _ptr(env_mean), _ptr(_ESA_WS[dev.index]),
                                            _stream()), "mtfjsp_enc_esa_mach_stats")
        Wf = torch.empty((128, 16), dtype=torch.float32, device=dev)
        Wp = torch.empty_like(Wf)
        bp = torch.empty(128, dtype=torch.float32, device=dev)
        b0f = torch.empty_like(bp)
        check(lib.mtfjsp_enc_esa_mach_fold(_ptr(moments), B * M, _ptr(w["m_fea_1_fcl.weight"]), _ptr(w["m_fea_2_fcl.weight"]),
                                           _ptr(w["bn.weight"]), _ptr(w["bn.bias"]), 1e-5, _ptr(w["m_policy.linears.0.weight"]),
                                           _ptr(w["m_policy.linears.0.bias"]), _ptr(Wf), _ptr(Wp), _ptr(bp), _ptr(b0f), _stream()),
              "mtfjsp_enc_esa_mach_fold")
        pooled = linear_tf32(env_mean, Wp, bp)
        bias = self._env_bias(pooled, h_pooled_o, b0f)
        w2 = self._derived("esa_w2", lambda: w["m_policy.linears.2.weight"].reshape(-1))
        s = torch.empty((B, M), dtype=torch.float32, device=dev)
        check(lib.mtfjsp_enc_esa_mach_head_tf32(_ptr(f1), _ptr(f2), B, M, _ptr(Wf), _ptr(bias), _ptr(w["m_policy.linears.1.weight"]),
                                                _ptr(w["m_policy.linears.1.bias"]), _ptr(w2), _ptr(w["m_policy.linears.2.bias"]),
                                                _ptr(s), _stream()), "mtfjsp_enc_esa_mach_head_tf32")
        return s, pooled


def global_critic_keys(hidden=128, in_dim=12):
    """state_dict layout of Global_Critic_JointAction_GAT (model/actor_critic.py:506-585); no checkpoint of it is
    shipped, the layout is pinned against the reference module by tests/golden/gen_ppo_golden.py."""
    H = hidden
    k = {n: s for n, s in job_actor_keys(hidden, in_dim).items() if n.startswith("encoder.")}
    for n, s in (("weight", (H,)), ("bias", (H,)), ("running_mean", (H,)), ("running_var", (H,)), ("num_batches_tracked", ())):
        k["bn." + n] = s
    k["m_fea_1_fcl.weight"] = (H, 6); k["m_fea_2_fcl.weight"] = (H, 8)
    k["gat_layer.W"] = (H, H); k["gat_layer.a"] = (1, 2 * H, 1)
    k["fcl_pooling.weight"] = (H, H)
    k["critic.linears.0.weight"] = (H, 2 * H); k["critic.linears.0.bias"] = (H,)
    k["critic.linears.1.weight"] = (H, H); k["critic.linears.1.bias"] = (H,)
    k["critic.linears.2.weight"] = (4, H); k["critic.linears.2.bias"] = (4,)
    return k


class GlobalCritic(_GraphEncoder, _MachineTrunk):
    """Forward of Global_Critic_JointAction_GAT (model/actor_critic.py:587-751): graph encoder over the op nodes,
    machine trunk over the two machine feature sets, 4 values (mk, pt, tt, idle) from the two pooled embeddings."""

    def __init__(self, state_dict, n_job, n_machine, hidden=128, in_dim=12, device=None, trainable=False):
        self.J, self.M, self.N, self.H = n_job, n_machine, n_job * n_machine, hidden
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.w = _Params(global_critic_keys(hidden, in_dim), state_dict, self.device, trainable)
        self.precision = "fp32"
        self._pending = None

    def parameters(self):
        return self.w.parameters()

    def state_dict(self):
        return self.w.state_dict()

    def forward(self, task_fea, adj_w, adj_src, machine_fea_1, machine_fea_2, groups=1, adj_dst=None):
        """-> v [B,4].  (The candidate features the reference gathers at :650-655 are not used by its value head.)"""
        pooled_o, _ = self.encode(task_fea, adj_w, adj_src, groups, adj_dst)
        _, pooled_m = self.trunk(machine_fea_1, machine_fea_2, groups)
        return _mlp3_tanh(self.w, "critic.", torch.cat((pooled_m, pooled_o), dim=-1))    # actor_critic.py:737-750
