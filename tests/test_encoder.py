"""Encoder side (SURVEY.md 8 a13): state_dict compatibility with the shipped checkpoints (CPU) and forward parity of
JobActor / MachineActor on the device against golden outputs of the reference modules
(tests/golden/gen_encoder_golden.py), fed from the CUDA environment's native observation layout.
Tolerance: FP32 (rtol 2e-4, atol 2e-5) -- the reference runs these layers in float32 as well."""
import importlib
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_state_dict_layout_matches_shipped_checkpoints():
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    tab = json.load(open(os.path.join(GOLD, "shipped_checkpoint_keys.json")))
    job = {k: list(v) for k, v in enc.job_actor_keys(128).items()}
    mch = {k: list(v) for k, v in enc.machine_actor_keys(128).items()}
    assert job == tab["PPO_operation_actor_J6M6E2_1000.pth"]
    assert mch == tab["PPO_machine_actor_J6M6E2_1000.pth"]


@pytest.mark.gpu
@pytest.mark.parametrize("H,precision", [(128, "fp32"), (32, "fp32"), (128, "tf32")])
def test_actor_forward_matches_reference_modules(H, precision):
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    g = np.load(os.path.join(GOLD, "replay_j6m6_ls_esa.npz"))
    e = np.load(os.path.join(GOLD, "encoder_golden.npz"))
    J, M, E = int(g["J"]), int(g["M"]), int(g["E"])
    B = g["t"].shape[0]
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    env.load(g["t"], g["p"], g["transT"], g["edge"])
    env.scaler_init()
    env.reset(g["weights"][0])
    env.obs(1)
    job = enc.JobActor(enc.seeded_state_dict(enc.job_actor_keys(H), 11), J, M, hidden=H, precision=precision)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(H), 12), M, hidden=H, precision=precision)
    dev = env.device
    i32 = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.int32)).to(dev)
    # fp32: the reference's own arithmetic; tf32: 10-bit-mantissa operands through 6 GEMMs and 6 batch norms
    rt, at = (2e-4, 2e-5) if precision == "fp32" else (3e-2, 5e-3)
    close = lambda a, b, name: np.testing.assert_allclose(a.cpu().numpy(), b, rtol=rt, atol=at, err_msg=name)
    cur = -1
    for tag in ("init", "s05", "s20", "s34"):
        k = "H%d_%s_" % (H, tag)
        s = int(e[k + "step"])
        while cur < s:  # replay the dump's actions up to step s
            cur += 1
            act = g["actions"][0, cur]
            env.step_obs(i32(act[:, 0]), i32(act[:, 1]), 1)
        hgm = None if e[k + "hgm_in"].size == 0 else torch.tensor(e[k + "hgm_in"]).to(dev)
        ti, ai, la, prob, pooled, jv = job.forward(env.task_fea, env.adj_w, env.adj_src, env.candidate, hgm,
                                                   env.job_mask, greedy=True)
        close(prob, e[k + "prob"], "job prob " + tag)
        close(pooled, e[k + "pooled"], "job pooled " + tag)
        close(jv, e[k + "job_v"], "job value " + tag)
        if precision == "fp32":
            np.testing.assert_array_equal(ti.cpu().numpy(), e[k + "task_index"])
        nxt = g["actions"][0, s + 1]
        m1, mmask = env.mfea1(i32(nxt[:, 0]))
        np.testing.assert_array_equal(mmask.cpu().numpy().astype(bool), e[k + "mmask"])
        mp, hp, mv = mch.forward(m1, env.mach_fea, torch.tensor(e[k + "pooled"]).to(dev), mmask)
        # the machine side normalises over only B*M = 24 rows here: TF32 operand rounding is amplified by the tiny
        # batch statistics, so the tf32 wiring check is looser (the GEMM kernel itself is checked to 2e-5 below)
        mclose = close if precision == "fp32" else (
            lambda a, b, name: np.testing.assert_allclose(a.cpu().numpy(), b, rtol=5e-2, atol=5e-2, err_msg=name))
        mclose(mp, e[k + "mch_prob"], "machine prob " + tag)
        mclose(hp, e[k + "mch_pooled"], "machine pooled " + tag)
        mclose(mv, e[k + "mch_v"], "machine value " + tag)


@pytest.mark.gpu
def test_aggregate_kernel_matches_dense_fp64_reference():
    """gcn_mlp.py:125-149 forms the neighbourhood mean in FP64; the kernel is FP32 (see mtfjsp_encoder.cu header)."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    B, J, M, E = 64, 10, 10, 3
    d = ins.synthetic_instances(0, B, J, M, E, 3)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 3))
    for s in range(57):
        env.random_step(seed=1)
    A = env.dense_adj(torch.float64)                       # [B,N,N], adj[dst,src], diagonal 1 (reference layout)
    for C in (12, 128):
        h = torch.randn(B, J * M, C, device=env.device)
        ref = torch.bmm(A, h.double()) / (A != 0).sum(-1, keepdim=True).double()   # gcn_mlp.py:125-149
        out = enc.aggregate(h, env.adj_w, env.adj_src)
        # FP32 fused multiply-adds: within 3 FP32 ulp of the magnitude sum |A| |h| / deg of the reference FP64 value
        bound = 3 * 2.0 ** -24 * (torch.bmm(A.abs(), h.double().abs()) / (A != 0).sum(-1, keepdim=True).double()) + 1e-30
        assert bool(((out.double() - ref).abs() <= bound).all()), float(((out.double() - ref).abs() / bound).max())
        pm = enc.graph_mean(h)
        np.testing.assert_allclose(pm.cpu().numpy(), h.mean(1).cpu().numpy(), rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("K,rows,affine", [(128, 128, False), (128, 1000, True), (12, 333, False), (12, 4096 + 17, True),
                                           (128, 128 * 300 + 5, True), (64, 777, True),
                                           # every K class (16, 32, 64, 128), K below the class, K not a multiple of 8
                                           (4, 1, True), (8, 127, False), (16, 129, True), (20, 333, False), (32, 127, True),
                                           (36, 1, False), (60, 129, True), (68, 777, False), (100, 127, True), (124, 4096 + 17, True),
                                           # one row either side of the switch to the TMA operand at K = 128
                                           (128, 4095, True), (128, 4096, False), (128, 4096, True)])
def test_tcgen05_linear_matches_fp32_matmul(K, rows, affine):
    """Fused linear layer on the tensor cores (TF32 operands, FP32 accumulate) against an FP64 matmul of the
    TF32-rounded operands (tight) and against plain FP32 (TF32 tolerance, 10-bit mantissa).  Every instantiation of the
    cp.async kernel (K padded to 16, 32, 64, 128, the padding zero-filled) and the TMA kernel (K = 128, rows >= 4,096)."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + rows)
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = torch.randn(128, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(128, device="cuda", generator=g)
    sc = sh = None
    xin = x
    if affine:
        sc = torch.rand(K, device="cuda", generator=g) + 0.5
        sh = torch.randn(K, device="cuda", generator=g) * 0.3
        xin = torch.relu((x.double() * sc.double() + sh.double()).float())  # the kernel's prologue is a fused multiply-add
    stats = torch.zeros(256, dtype=torch.float64, device="cuda")
    z = enc.linear_tf32(x, W, b, sc, sh, relu=affine, stats=stats)
    torch.cuda.synchronize()

    def tf32(t):  # round-to-nearest-away on the 13 dropped mantissa bits (cvt.rna.tf32.f32)
        i = t.contiguous().view(torch.int32)
        return ((i + 0x1000) & ~0x1FFF).view(torch.float32)

    ref_t = (tf32(xin).double() @ tf32(W).double().T + b.double())
    ref_f = xin.double() @ W.double().T + b.double()
    np.testing.assert_allclose(z.double().cpu().numpy(), ref_t.cpu().numpy(), rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(z.double().cpu().numpy(), ref_f.cpu().numpy(), rtol=5e-3, atol=5e-3)
    np.testing.assert_allclose(stats[:128].cpu().numpy(), z.double().sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)
    np.testing.assert_allclose(stats[128:].cpu().numpy(), (z.double() ** 2).sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)
    if rows == 1:  # torch's batch_norm needs two rows per channel
        return
    scale, shift = enc.bn_finalize(stats, rows, torch.ones(128, device="cuda"), torch.zeros(128, device="cuda"))
    bn = torch.nn.functional.batch_norm(z, None, None, None, None, True, 0.0, 1e-5)
    np.testing.assert_allclose((z * scale + shift).cpu().numpy(), bn.cpu().numpy(), rtol=1e-3, atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("B,rpe,nodes,affine,per_env_bias", [(7, 6, 36, True, True), (1000, 6, 36, True, True),
                                                            (148 * 128 * 2 // 6 + 3, 6, 0, False, True), (333, 10, 100, True, False),
                                                            (50, 20, 0, False, False), (500, 6, 0, "norelu", True)])
def test_fused_policy_head_matches_the_separate_launches(B, rpe, nodes, affine, per_env_bias):
    """mtfjsp_enc_head_tf32 (gather + BatchNorm/ReLU prologue + Linear + per-env bias + tanh + Linear + tanh + dot, one
    launch, intermediate kept on the SM) against an FP64 evaluation with TF32-rounded GEMM operands (tight) and against
    plain FP32 (TF32 tolerance)."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(B * 31 + rpe)
    H = 128
    rows = B * rpe
    if nodes:
        x = torch.randn(B, nodes, H, device="cuda", generator=g)
        cand = torch.randint(0, nodes, (B, rpe), device="cuda", generator=g, dtype=torch.int32)
        per_row = torch.gather(x, 1, cand.long().unsqueeze(-1).expand(-1, rpe, H)).reshape(rows, H)
    else:
        x = torch.randn(rows, H, device="cuda", generator=g)
        cand = None
        per_row = x
    sc = sh = None
    if affine:
        sc = torch.rand(H, device="cuda", generator=g) + 0.5
        sh = torch.randn(H, device="cuda", generator=g) * 0.3
        per_row = (per_row.double() * sc.double() + sh.double()).float()
        if affine != "norelu":
            per_row = torch.relu(per_row)
    Wa = torch.randn(H, H, device="cuda", generator=g) / H ** 0.5
    W1 = torch.randn(H, H, device="cuda", generator=g) / H ** 0.5
    b1 = torch.randn(H, device="cuda", generator=g) * 0.2
    w2 = torch.randn(H, device="cuda", generator=g) / H ** 0.5
    b2 = torch.randn(1, device="cuda", generator=g)
    bias = torch.randn(B if per_env_bias else 1, H, device="cuda", generator=g) * 0.5
    out = enc.head_tf32(x, cand, B, rpe, nodes, sc, sh, Wa, bias, W1, b1, w2, b2, relu=affine != "norelu")
    torch.cuda.synchronize()

    def tf32(t):
        i = t.contiguous().view(torch.int32)
        return ((i + 0x1000) & ~0x1FFF).view(torch.float32)

    brow = bias.double().repeat_interleave(rpe, dim=0) if per_env_bias else bias.double()

    def chain(rnd):
        z = torch.tanh((rnd(per_row).double() @ rnd(Wa).double().T + brow).float())
        z = torch.tanh((rnd(z).double() @ rnd(W1).double().T + b1.double()).float())
        return (z.double() @ w2.double() + b2.double()).view(B, rpe)

    np.testing.assert_allclose(out.double().cpu().numpy(), chain(tf32).cpu().numpy(), rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(out.double().cpu().numpy(), chain(lambda t: t).cpu().numpy(), rtol=1e-2, atol=1e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,affine", [(5, 36, True), (1000, 36, True), (148 * 3 * 2 + 1, 36, False), (77, 100, True), (40, 128, True),
                                        (300, 60, False)])
def test_fused_aggregation_and_layer_match_the_two_kernels(B, N, affine):
    """mtfjsp_enc_aggregate_linear_tf32 (the weighted neighbourhood mean applied to the product rows in the epilogue,
    tiles of whole envs) against aggregate -> linear in FP64 (TF32-rounded GEMM operands; the sum is taken after the
    product, so the comparison carries TF32 rounding of the single rows: 2e-3) and against the two separate kernels."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(B * 7 + N)
    H = 128
    h = torch.randn(B, N, H, device="cuda", generator=g)
    M = 6 if N == 36 else (10 if N == 100 else 4)   # ops per job: the first op of a job has no job predecessor
    adj_w = torch.rand(B, N, 2, device="cuda", generator=g) + 0.5
    adj_w[:, ::M, 0] = 0.0
    adj_src = torch.randint(-1, N, (B, N), device="cuda", generator=g, dtype=torch.int16)
    adj_w[..., 1] = torch.where(adj_src >= 0, adj_w[..., 1], torch.zeros_like(adj_w[..., 1]))
    drop = torch.rand(B, N, device="cuda", generator=g) < 0.3   # some rows without a job predecessor at all
    adj_w[..., 0] = torch.where(drop, torch.zeros_like(adj_w[..., 0]), adj_w[..., 0])
    W = torch.randn(H, H, device="cuda", generator=g) / H ** 0.5
    b = torch.randn(H, device="cuda", generator=g)
    sc = sh = None
    if affine:
        sc = torch.rand(H, device="cuda", generator=g) + 0.5
        sh = torch.randn(H, device="cuda", generator=g) * 0.3
    stats = torch.zeros(256, dtype=torch.float64, device="cuda")
    z = enc.aggregate_linear_tf32(h, adj_w, adj_src, W, b, sc, sh, relu=affine, stats=stats)
    assert z is not None
    torch.cuda.synchronize()
    pooled = enc.aggregate(h, adj_w, adj_src, sc, sh, relu=affine).reshape(B * N, H)
    ref = pooled.double() @ W.double().T + b.double()
    np.testing.assert_allclose(z.double().cpu().numpy(), ref.cpu().numpy(), rtol=5e-3, atol=5e-3)
    two = enc.linear_tf32(pooled, W, b)
    np.testing.assert_allclose(z.cpu().numpy(), two.cpu().numpy(), rtol=5e-3, atol=5e-3)
    np.testing.assert_allclose(stats[:128].cpu().numpy(), z.double().sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)
    np.testing.assert_allclose(stats[128:].cpu().numpy(), (z.double() ** 2).sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [6, 10, 30])
def test_selection_kernel_softmax_draws_and_log_probabilities(R):
    """mtfjsp_enc_select against torch: prob = masked softmax, greedy = arg-max, log_a = log prob[action], task = the
    candidate behind the action; draws never pick an excluded entry, follow the distribution (chi-square-like bound on
    65,536 draws of one distribution) and change when the device step counter advances."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(R)
    B = 4099
    scores = torch.randn(B, R, device="cuda", generator=g) * 2
    mask = torch.rand(B, R, device="cuda", generator=g) < 0.4
    mask[:, 0] &= ~mask.all(dim=1)      # at least one open entry per row
    cand = torch.randint(0, 600, (B, R), device="cuda", generator=g, dtype=torch.int32)
    ref = torch.softmax((scores * 10.0).masked_fill(mask, float("-inf")), dim=-1)
    prob, a, la, task = enc.select(scores, mask, cand, 10.0, True, None, 0)
    np.testing.assert_allclose(prob.cpu().numpy(), ref.cpu().numpy(), rtol=2e-6, atol=1e-7)
    assert torch.equal(a, ref.argmax(dim=-1))
    np.testing.assert_allclose(la.cpu().numpy(), torch.log(ref.gather(1, a[:, None])[:, 0]).cpu().numpy(), rtol=1e-5, atol=1e-6)
    assert torch.equal(task, cand.long().gather(1, a[:, None])[:, 0])
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    p1, a1, la1, t1 = enc.select(scores, mask, cand, 10.0, False, (7, counter), 0)
    assert not bool(mask.gather(1, a1[:, None]).any())                     # never an excluded entry
    np.testing.assert_allclose(la1.cpu().numpy(), torch.log(p1.gather(1, a1[:, None])[:, 0]).cpu().numpy(), rtol=1e-5, atol=1e-6)
    p1b, a1b, _, _ = enc.select(scores, mask, cand, 10.0, False, (7, counter), 0)
    assert torch.equal(a1, a1b)                                            # same key, same draw
    counter.add_(1)
    _, a2, _, _ = enc.select(scores, mask, cand, 10.0, False, (7, counter), 0)
    _, a3, _, _ = enc.select(scores, mask, cand, 10.0, False, (7, counter), 1)
    soft = enc.select(scores, mask, cand, 1.0, False, (7, counter), 0)[1]
    assert not torch.equal(soft, a2) and not torch.equal(a2, a3)           # step counter, stream id and scale all matter
    one = torch.randn(1, R, device="cuda", generator=g).expand(65536, R).contiguous()
    nomask = torch.zeros(65536, R, dtype=torch.bool, device="cuda")
    pd, ad, _, _ = enc.select(one, nomask, None, 1.0, False, (11, counter), 0)
    freq = torch.bincount(ad, minlength=R).double() / 65536
    err = (freq - pd[0].double()).abs() / torch.sqrt(pd[0].double() * (1 - pd[0].double()) / 65536 + 1e-12)
    assert float(err.max()) < 5.0, (freq, pd[0])                           # within five standard deviations per entry


@pytest.mark.gpu
@pytest.mark.parametrize("R", [5, 64, 1000, 64 * 148 * 2 + 17])
def test_fused_machine_trunk_matches_the_fp64_chain_on_tf32_operands(R):
    """mtfjsp_enc_gat_trunk_tf32 (input projections + three GAT layers + node-set mean, one launch, 128 machines per SM)
    against the same chain in FP64 with TF32-rounded GEMM operands (tight) and plain FP32 (TF32 tolerance over three
    layers)."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(R)
    H = 128
    f1 = torch.randn(R, 6, device="cuda", generator=g)
    f2 = torch.randn(R, 8, device="cuda", generator=g)
    W1p = torch.randn(H, 6, device="cuda", generator=g) / 6 ** 0.5
    W2p = torch.randn(H, 8, device="cuda", generator=g) / 8 ** 0.5
    Wt = (torch.randn(H, H, device="cuda", generator=g) / H ** 0.5).contiguous()
    a_src = torch.randn(H, device="cuda", generator=g) / H ** 0.5
    a_dst = torch.randn(H, device="cuda", generator=g) / H ** 0.5
    stats = torch.zeros(256, dtype=torch.float64, device="cuda")
    out = enc.gat_trunk_tf32(f1, f2, W1p, W2p, Wt, a_src, a_dst, stats)
    torch.cuda.synchronize()
    np.testing.assert_allclose(stats[:128].cpu().numpy(), out.double().sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)
    np.testing.assert_allclose(stats[128:].cpu().numpy(), (out.double() ** 2).sum(0).cpu().numpy(), rtol=1e-5, atol=1e-3)

    def tf32(t):
        i = t.contiguous().view(torch.int32)
        return ((i + 0x1000) & ~0x1FFF).view(torch.float32)

    def chain(rnd):
        h1, h2 = F.linear(f1, W1p), F.linear(f2, W2p)
        for layer in range(3):
            t1 = (rnd(h1).double() @ rnd(Wt).double().T).float()
            t2 = (rnd(h2).double() @ rnd(Wt).double().T).float()
            e11 = F.leaky_relu(t1 @ a_src + t1 @ a_dst, 0.2)
            e12 = F.leaky_relu(t1 @ a_src + t2 @ a_dst, 0.2)
            att = torch.softmax(torch.stack((e11, e12), dim=-1), dim=-1)
            h1, h2 = att[:, 0:1] * t1 + att[:, 1:2] * t2, t2
            if layer < 2:
                h1, h2 = F.elu(h1), F.elu(h2)
        return 0.5 * (h1 + h2)

    np.testing.assert_allclose(out.cpu().numpy(), chain(tf32).cpu().numpy(), rtol=3e-3, atol=3e-3)  # a flipped TF32 rounding = 5e-4
    np.testing.assert_allclose(out.cpu().numpy(), chain(lambda t: t).cpu().numpy(), rtol=3e-2, atol=3e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("K,rows", [(128, 64), (128, 1000), (12, 333), (12, 64 * 200 + 17), (128, 64 * 148 * 3 + 5),
                                    (64, 777), (32, 4096),
                                    # K below its class (4 / 16, 20 / 32, 36 / 64, 100 / 128), one partial 64-row stage
                                    (4, 1), (16, 63), (20, 65), (36, 1), (100, 63), (100, 65), (4, 64 * 148 + 3)])
def test_tcgen05_weight_gradient_matches_fp64_product(K, rows):
    """dW = dY^T X and db = column sums of dY on the tensor cores (TF32 operands, FP32 accumulate over the rows of a
    CTA, fixed-order FP32 sum of the CTA partials) against the FP64 product of the TF32-rounded operands (tight:
    FP32 accumulation error only) and of the unrounded ones (TF32 tolerance); two runs must agree bit for bit."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + rows)
    x = torch.randn(rows, K, device="cuda", generator=g)
    gz = torch.randn(rows, 128, device="cuda", generator=g)
    dW, db = enc.wgrad_tf32(gz, x)
    dW2, db2 = enc.wgrad_tf32(gz, x)
    torch.cuda.synchronize()
    assert torch.equal(dW, dW2) and torch.equal(db, db2)

    def tf32(t):
        i = t.contiguous().view(torch.int32)
        return ((i + 0x1000) & ~0x1FFF).view(torch.float32)

    ref_t = tf32(gz).double().T @ tf32(x).double()
    ref_f = gz.double().T @ x.double()
    scale = float(rows) ** 0.5  # entries are sums of `rows` products of unit normals
    np.testing.assert_allclose(dW.double().cpu().numpy() / scale, ref_t.cpu().numpy() / scale, rtol=0, atol=2e-5)
    if rows >= 64:
        np.testing.assert_allclose(dW.double().cpu().numpy() / scale, ref_f.cpu().numpy() / scale, rtol=0, atol=3e-3)
    else:  # too few rows to average the operand rounding: each operand within 2^-11 of its TF32 value
        bound = 2.0 ** -10 * (gz.double().abs().T @ x.double().abs()) + 1e-6
        assert bool(((dW.double() - ref_f).abs() <= bound).all())
    np.testing.assert_allclose(db.double().cpu().numpy() / scale, gz.double().sum(0).cpu().numpy() / scale, rtol=0, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [12, 128])
def test_tcgen05_training_linear_gradients_match_autograd(K):
    """linear_train(tf32=True): forward, input gradient and weight / bias gradients against torch autograd of F.linear."""
    torch = pytest.importorskip("torch")
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(K)
    rows = 5000
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = (torch.randn(128, K, device="cuda", generator=g) / K ** 0.5)
    b = torch.randn(128, device="cuda", generator=g)
    gy = torch.randn(rows, 128, device="cuda", generator=g)
    outs = []
    for tf in (False, True):
        xi, Wi, bi = x.clone().requires_grad_(True), W.clone().requires_grad_(True), b.clone().requires_grad_(True)
        z = enc.linear_train(xi, Wi, bi, tf)
        z.backward(gy)
        outs.append((z.detach(), xi.grad, Wi.grad, bi.grad))
    for a, r, name, sc in zip(outs[1], outs[0], ("z", "dx", "dW", "db"), (1.0, 1.0, rows ** 0.5, rows ** 0.5)):
        np.testing.assert_allclose(a.cpu().numpy() / sc, r.cpu().numpy() / sc, rtol=0, atol=6e-3, err_msg=name)


@pytest.mark.gpu
def test_gat_attend_kernel_matches_torch():
    """gat_attend (the GAT layer after its projection) against the torch expression it replaces
    (actor_critic.py:400-420, model/gat.py:82-159), FP32 tolerance."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(7)
    rn = lambda *sh: torch.randn(*sh, device="cuda", generator=g)
    close = lambda a, b, tol=2e-5: np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=tol, atol=tol)
    R = 1003
    t, a_src, a_dst = rn(2 * R, 128), rn(128) * 0.1, rn(128) * 0.1
    t1, t2 = t[:R], t[R:]
    e11 = F.leaky_relu(t1 @ a_src + t1 @ a_dst, 0.2)
    e12 = F.leaky_relu(t1 @ a_src + t2 @ a_dst, 0.2)
    att = torch.softmax(torch.stack((e11, e12), -1), -1)
    h1, h2 = att[:, 0:1] * t1 + att[:, 1:2] * t2, t2
    close(enc.gat_attend(t, a_src, a_dst, 0), torch.cat((h1, h2), 0), 1e-4)
    close(enc.gat_attend(t, a_src, a_dst, 1), torch.cat((F.elu(h1), F.elu(h2)), 0), 1e-4)
    close(enc.gat_attend(t, a_src, a_dst, 2), torch.stack((h1, h2), 1).mean(1), 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gat_attend_backward_matches_torch_autograd(mode):
    """gat_attend_train (forward kernel + hand-written backward) against autograd of the torch expression it replaces."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
    g = torch.Generator(device="cuda").manual_seed(3 + mode)
    R = 2051
    t0 = torch.randn(2 * R, 128, device="cuda", generator=g)
    as0 = torch.randn(128, device="cuda", generator=g) * 0.1
    ad0 = torch.randn(128, device="cuda", generator=g) * 0.1

    def ref(t, a_src, a_dst):
        t1, t2 = t[:R], t[R:]
        e11 = F.leaky_relu(t1 @ a_src + t1 @ a_dst, 0.2)
        e12 = F.leaky_relu(t1 @ a_src + t2 @ a_dst, 0.2)
        att = torch.softmax(torch.stack((e11, e12), -1), -1)
        h1, h2 = att[:, 0:1] * t1 + att[:, 1:2] * t2, t2
        if mode == 0:
            return torch.cat((h1, h2), 0)
        if mode == 1:
            return torch.cat((F.elu(h1), F.elu(h2)), 0)
        return torch.stack((h1, h2), 1).mean(1)

    outs = []
    for fn in (ref, lambda t, a, b: enc.gat_attend_train(t, a, b, mode)):
        t, a, b = t0.clone().requires_grad_(True), as0.clone().requires_grad_(True), ad0.clone().requires_grad_(True)
        y = fn(t, a, b)
        gy = torch.randn(y.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(99))
        y.backward(gy)
        outs.append((y.detach(), t.grad, a.grad, b.grad))
    for x, r, name, sc in zip(outs[1], outs[0], ("y", "dt", "da_src", "da_dst"), (1.0, 1.0, R ** 0.5, R ** 0.5)):
        np.testing.assert_allclose(x.cpu().numpy() / sc, r.cpu().numpy() / sc, rtol=0, atol=2e-4, err_msg=name)
