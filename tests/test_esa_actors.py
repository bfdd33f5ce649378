"""ESA-PPO baseline actors (esa_Operation_Actor_Critic / esa_Machine_Actor, model/actor_critic.py:945-1404): state_dict
layout of the shipped tester/ESWA_MPPO checkpoints, the algebra of the folded machine actor, parity with the reference
modules (tests/golden/gen_esa_golden.py), the three machine-actor kernels, and greedy validation with the shipped J6M6E2
checkpoints against result CSV row 14 (`ESA-PPO`)."""
import importlib
import json
import os
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

GOLD = os.path.join(os.path.dirname(__file__), "golden")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")


def _objective(x):
    return 0.4 * x[:, 0] + 0.4 * (x[:, 1] + x[:, 3]) + 0.2 * x[:, 2]


def test_key_tables_match_all_shipped_esa_checkpoints():
    tab = json.load(open(os.path.join(GOLD, "shipped_esa_checkpoint_keys.json")))
    assert len(tab) == 12
    sizes = set()
    for name, keys in tab.items():
        want = enc.esa_job_actor_keys(128) if "_operation_actor_" in name else enc.esa_machine_actor_keys(128)
        assert keys == {k: list(v) for k, v in want.items()}, name
        sizes.add(name.split("_")[-2])
    assert sizes == {"J6M6E2", "J10M6E2", "J20M6E3", "J10M10E2", "J15M10E2", "J20M10E5"}


def _fold64(f1, f2, W1, W2, gamma, beta, W0, b0, eps=1e-5):
    """The fold restated in torch: moments -> BatchNorm affine -> folded first layer, per-env pooled embedding."""
    R = f1.shape[0]
    H = W1.shape[0]
    out = []
    for f, W in ((f1, W1), (f2, W2)):
        mu = f.sum(0) / R
        cov = f.T @ f / R - torch.outer(mu, mu)
        var = ((W @ cov) * W).sum(1).clamp_min(0)
        sc = gamma / torch.sqrt(var + eps)
        out.append((W * sc[:, None], beta - (W @ mu) * sc))
    (A1, sh1), (A2, sh2) = out
    Wf = torch.cat((W0[:, :H] @ A1, W0[:, H:2 * H] @ A2), 1)
    b0f = b0 + W0[:, :H] @ sh1 + W0[:, H:2 * H] @ sh2
    return Wf, b0f, torch.cat((A1, A2), 1) / 2, (sh1 + sh2) / 2


def test_fold_equals_literal_batchnorm_concat_and_first_layer_fp64():
    """W0 cat(BN(f1 W1^T), BN(f2 W2^T), pooled, h_o) + b0 with batch statistics == [f1|f2] Wf^T + b0f + W0c pooled + W0d h_o,
    pooled == mean_m([f1|f2]) Wp^T + bp; FP64, features with a large common offset and one constant column."""
    g = torch.Generator().manual_seed(5)
    B, M, H = 37, 10, 128
    R = B * M
    d = torch.float64
    f1 = torch.rand((R, 6), generator=g, dtype=d) * 3 + 20.0
    f2 = torch.randn((R, 8), generator=g, dtype=d)
    f2[:, 5] = 0.75
    sd = enc.seeded_state_dict(enc.esa_machine_actor_keys(H), 3)
    W1, W2 = sd["m_fea_1_fcl.weight"].double(), sd["m_fea_2_fcl.weight"].double()
    gamma, beta = sd["bn.weight"].double(), sd["bn.bias"].double()
    W0, b0 = sd["m_policy.linears.0.weight"].double(), sd["m_policy.linears.0.bias"].double()
    h_o = torch.randn((B, H), generator=g, dtype=d)
    bn = lambda x: torch.nn.functional.batch_norm(x, None, None, gamma, beta, True, 0.0, 1e-5)
    h1, h2 = bn(f1 @ W1.T).view(B, M, H), bn(f2 @ W2.T).view(B, M, H)
    pooled = (h1.mean(1) + h2.mean(1)) / 2
    x = torch.cat((h1, h2, pooled[:, None].expand_as(h1), h_o[:, None].expand_as(h1)), -1)
    lit = x @ W0.T + b0
    Wf, b0f, Wp, bp = _fold64(f1, f2, W1, W2, gamma, beta, W0, b0)
    f = torch.cat((f1, f2), 1)
    pooled_f = f.view(B, M, 14).mean(1) @ Wp.T + bp
    np.testing.assert_allclose(pooled_f.numpy(), pooled.numpy(), rtol=1e-10, atol=1e-10)
    fold = (f @ Wf.T).view(B, M, H) + (b0f + pooled_f @ W0[:, 2 * H:3 * H].T + h_o @ W0[:, 3 * H:].T)[:, None]
    np.testing.assert_allclose(fold.numpy(), lit.numpy(), rtol=1e-10, atol=1e-10)


def test_machine_actor_fp32_matches_reference_module_on_cpu():
    """The literal FP32 form needs no kernel with one BatchNorm group: checked against the reference module here too."""
    g = np.load(os.path.join(GOLD, "replay_j6m6_ls_esa.npz"))
    e = np.load(os.path.join(GOLD, "esa_golden.npz"))
    for H in (128, 32):
        mch = enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(H), 22), 6, hidden=H, device="cpu")
        for s in (5, 20):
            k = "H%d_s%02d_g1_" % (H, s)
            with torch.no_grad():
                mp, hp, mv = mch.forward(torch.tensor(g["mfea1"][0, s + 1]), torch.tensor(g["mfea2"][0, s]), torch.tensor(e[k + "pooled"]),
                                         torch.tensor(e["H%d_s%02d_mmask" % (H, s)]))
                lg, _, _ = mch.forward(torch.tensor(g["mfea1"][0, s + 1]), torch.tensor(g["mfea2"][0, s]), torch.tensor(e[k + "pooled"]),
                                       None, return_logits=True)
            for a, name in ((mp, "mch_prob"), (hp, "mch_pooled"), (mv, "mch_v"), (lg, "mch_logits")):
                np.testing.assert_allclose(a.numpy(), e[k + name], rtol=2e-4, atol=2e-5, err_msg=k + name)


def test_ppo_collect_refuses_esa_actors():
    ppo = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.ppo")
    ro = types.SimpleNamespace(env=types.SimpleNamespace(N=36), job=object.__new__(enc.EsaJobActor), mch=None)
    with pytest.raises(TypeError, match="ESA"):
        ppo.collect(ro, [np.array([0.4, 0.4, 0.2])])


# --------------------------------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("H,precision", [(128, "fp32"), (32, "fp32"), (128, "tf32")])
def test_actors_match_reference_modules(H, precision):
    """Both ESA actors against the reference modules fed from the CUDA env's native observations; case gB: per-instance
    BatchNorm groups (fp32) against B separate batch-1 reference calls.  Tolerances of
    test_encoder.py::test_actor_forward_matches_reference_modules (the machine side normalises over only 24 rows).
    In case gB the machine BatchNorm sees 6 rows per group: columns whose 6 values nearly coincide have a variance near
    eps, where the grouped device kernel (FP64 sums) and PyTorch's CPU batch norm round differently; measured on a B200:
    one element of 24 off by 1.2e-4 (scores / 10) and one of 128 by 2.8e-5 (pooled), hence 1e-3 / 5e-4 there."""
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    g = np.load(os.path.join(GOLD, "replay_j6m6_ls_esa.npz"))
    e = np.load(os.path.join(GOLD, "esa_golden.npz"))
    J, M, E = int(g["J"]), int(g["M"]), int(g["E"])
    B = g["t"].shape[0]
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    env.load(g["t"], g["p"], g["transT"], g["edge"])
    env.scaler_init()
    env.reset(g["weights"][0])
    env.obs(1)
    job = enc.EsaJobActor(enc.seeded_state_dict(enc.esa_job_actor_keys(H), 21), J, M, hidden=H, precision=precision)
    mch = enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(H), 22), M, hidden=H, precision=precision)
    dev = env.device
    i32 = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.int32)).to(dev)
    rt, at = (2e-4, 2e-5) if precision == "fp32" else (3e-2, 5e-3)
    mrt, mat = (2e-4, 2e-5) if precision == "fp32" else (5e-2, 5e-2)
    cur = -1
    for s in (5, 20):
        while cur < s:
            cur += 1
            act = g["actions"][0, cur]
            env.step_obs(i32(act[:, 0]), i32(act[:, 1]), 1)
        hgm = torch.tensor(e["H%d_s%02d_hgm_in" % (H, s)]).to(dev)
        nxt = g["actions"][0, s + 1]
        m1, mmask = env.mfea1(i32(nxt[:, 0]))
        for case in ("g1", "gB") if precision == "fp32" else ("g1",):
            k = "H%d_s%02d_%s_" % (H, s, case)
            groups = B if case == "gB" else 1
            with torch.no_grad():
                prob, pooled, jv = job.evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, hgm, env.job_mask, groups=groups)
                h_o = torch.tensor(e[k + "pooled"]).to(dev)
                mp, hp, mv = mch.forward(m1, env.mach_fea, h_o, mmask, groups=groups)
                lg, _, _ = mch.forward(m1, env.mach_fea, h_o, mmask, groups=groups, return_logits=True)
            assert jv.shape == (B, 4) and mv.shape == (B, 2)
            for a, name, r, t in ((prob, "prob", rt, at), (pooled, "pooled", rt, at), (jv, "job_v", rt, at), (mp, "mch_prob", mrt, mat),
                                  (hp, "mch_pooled", mrt, mat), (mv, "mch_v", mrt, mat), (lg / 10, "mch_logits", mrt, mat)):
                ref = e[k + name] / (10 if name == "mch_logits" else 1)
                if case == "gB" and name.startswith("mch"):
                    r, t = 1e-3, 5e-4
                np.testing.assert_allclose(a.cpu().numpy(), ref, rtol=r, atol=t, err_msg=k + name)


def _tf32(t):  # round-to-nearest-away on the 13 dropped mantissa bits (cvt.rna.tf32.f32)
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _features(B, M, seed, const_col):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f1 = torch.rand((B * M, 6), generator=g, device="cuda") * 4 + 1
    f2 = torch.randn((B * M, 8), generator=g, device="cuda")
    if const_col:
        f2[:, 3] = 0.625
    return f1, f2


@pytest.mark.gpu
@pytest.mark.parametrize("B,M,const_col", [(5, 1, False), (32, 2, True), (100, 10, False), (6318, 6, True), (1895, 20, False),
                                           (11, 6, False)])
def test_esa_kernels_match_fp64(B, M, const_col):
    """mtfjsp_enc_esa_mach_stats (moments FP64, per-env means), mtfjsp_enc_esa_mach_fold (FP64 fold) and
    mtfjsp_enc_esa_mach_head_tf32 against FP64 evaluations: the head with TF32-rounded operands at the tolerance of
    test_encoder.py's head-kernel test; R = 5 .. 37,908 rows, M = 6 / 10 / 20 (envs straddle the 128-row tiles),
    a constant feature column (variance 0)."""
    lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib").lib()
    mch = enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 9), M, precision="tf32")
    w = mch.w
    f1, f2 = _features(B, M, B + M, const_col)
    R = B * M
    ws = torch.empty(int(lib.mtfjsp_enc_esa_mach_stats_workspace_doubles()), dtype=torch.float64, device="cuda")
    mom = torch.empty(114, dtype=torch.float64, device="cuda")
    em = torch.empty((B, 16), dtype=torch.float32, device="cuda")
    P = enc._ptr
    enc.check(lib.mtfjsp_enc_esa_mach_stats(P(f1), P(f2), B, M, P(mom), P(em), P(ws), enc._stream()), "stats")
    f = torch.cat((f1, f2), 1).double()
    want = torch.cat((f.sum(0), (f[:, :6].T @ f[:, :6]).reshape(-1), (f[:, 6:].T @ f[:, 6:]).reshape(-1)))
    np.testing.assert_allclose(mom.cpu().numpy(), want.cpu().numpy(), rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(em[:, :14].cpu().numpy(), f.view(B, M, 14).mean(1).cpu().numpy(), rtol=1e-6, atol=1e-7)
    assert (em[:, 14:] == 0).all()
    mom2 = torch.empty_like(mom)
    enc.check(lib.mtfjsp_enc_esa_mach_stats(P(f1), P(f2), B, M, P(mom2), P(em), P(ws), enc._stream()), "stats")
    assert torch.equal(mom, mom2)  # fixed-order reduction

    Wf, Wp = torch.empty((128, 16), device="cuda"), torch.empty((128, 16), device="cuda")
    bp, b0f = torch.empty(128, device="cuda"), torch.empty(128, device="cuda")
    enc.check(lib.mtfjsp_enc_esa_mach_fold(P(mom), R, P(w["m_fea_1_fcl.weight"]), P(w["m_fea_2_fcl.weight"]), P(w["bn.weight"]),
                                           P(w["bn.bias"]), 1e-5, P(w["m_policy.linears.0.weight"]), P(w["m_policy.linears.0.bias"]),
                                           P(Wf), P(Wp), P(bp), P(b0f), enc._stream()), "fold")
    d = lambda k: w[k].double()
    rWf, rb0f, rWp, rbp = _fold64(f[:, :6], f[:, 6:], d("m_fea_1_fcl.weight"), d("m_fea_2_fcl.weight"), d("bn.weight"), d("bn.bias"),
                                  d("m_policy.linears.0.weight"), d("m_policy.linears.0.bias"))
    for a, b in ((Wf[:, :14], rWf), (Wp[:, :14], rWp), (bp, rbp), (b0f, rb0f)):
        np.testing.assert_allclose(a.double().cpu().numpy(), b.cpu().numpy(), rtol=1e-5, atol=1e-5)
    assert (Wf[:, 14:] == 0).all() and (Wp[:, 14:] == 0).all()

    bias = torch.randn((B, 128), device="cuda") * 0.5
    W1, b1, b2 = w["m_policy.linears.1.weight"], w["m_policy.linears.1.bias"], w["m_policy.linears.2.bias"]
    w2 = w["m_policy.linears.2.weight"].reshape(-1).contiguous()
    out = torch.empty((B, M), device="cuda")
    enc.check(lib.mtfjsp_enc_esa_mach_head_tf32(P(f1), P(f2), B, M, P(Wf), P(bias), P(W1), P(b1), P(w2), P(b2), P(out), enc._stream()),
              "head")
    torch.cuda.synchronize()
    x = torch.cat((f1, f2, torch.zeros((R, 2), device="cuda")), 1)
    z = torch.tanh((_tf32(x).double() @ _tf32(Wf).double().T + bias.double().repeat_interleave(M, 0)).float())
    z = torch.tanh((_tf32(z).double() @ _tf32(W1).double().T + b1.double()).float())
    ref = 10 * (z.double() @ w2.double() + b2.double()).view(B, M)
    np.testing.assert_allclose(out.double().cpu().numpy() / 10, ref.cpu().numpy() / 10, rtol=2e-4, atol=2e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("B,M", [(4, 6), (1000, 6), (300, 10), (700, 20)])
def test_fused_machine_actor_matches_layer_by_layer(B, M, monkeypatch):
    """The fused tf32 machine actor (stats + fold + head) against MTFJSP_FUSED_ESA=0 (projections, BatchNorms and the
    split first layer as separate launches) and against the FP32 actor.  The two tf32 forms round different operands
    to TF32 (raw features vs. normalised embeddings), so they agree to TF32 accuracy, not bit for bit."""
    sd = enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 31)
    f1, f2 = _features(B, M, 7 * B + M, True)
    f1, f2 = f1.view(B, M, 6), f2.view(B, M, 8)
    h_o = torch.randn((B, 128), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
    mask = torch.zeros((B, M), dtype=torch.bool, device="cuda")
    res = {}
    with torch.no_grad():
        for name, prec, fused in (("fused", "tf32", True), ("layers", "tf32", False), ("fp32", "fp32", True)):
            monkeypatch.setattr(enc, "_FUSED_ESA", fused)
            mch = enc.EsaMachineActor(sd, M, precision=prec)
            res[name] = [t.cpu().numpy() for t in mch.forward(f1, f2, h_o, mask, return_logits=True)]
    for other in ("layers", "fp32"):
        for i, name in enumerate(("scores", "pooled", "machine_v")):
            a, b = res["fused"][i], res[other][i]
            np.testing.assert_allclose(a, b, rtol=1e-2, atol=1e-2 * max(1.0, np.abs(b).max()), err_msg="%s vs %s" % (name, other))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,min_same", [("fp32", 5), ("tf32", 10)])
def test_greedy_validation_with_shipped_esa_checkpoints_reproduces_csv_row_14(precision, min_same):
    """tester/ESWA_MPPO/esa_PPO_{operation,machine}_actor_J6M6E2_800.pth, greedy, the 100 shipped test instances, per-instance
    BatchNorm, through validate.greedy_validate unchanged.  The unmodified reference validation on CPU reproduces 100 / 100
    rows of the authors' CSV row 14 (esa_golden.npz ref_cpu).  Floors: fp32 >= that - 5, tf32 >= that - 10 instances
    bit-identical to the CSV; mean objective within 0.5 %.  Measured on a B200: fp32 100 / 100 identical to the CSV (and to
    the CPU reference), tf32 97 / 100 (DESIGN.md section 2)."""
    val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
    g = np.load(os.path.join(GOLD, "esa_golden.npz"))
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    inst = {k: pd[k] for k in ("t", "p", "transT", "edge")}
    sd_op, sd_m = val.load_actor_state_dicts(g, "esa")
    # the fixture holds the tensors the policy decisions read; the value heads and the machine actor's unread
    # gat_layer / fcl_pooling tensors are left out of it and stand in as zeros (greedy validation discards the values)
    kop, km = enc.esa_job_actor_keys(128), enc.esa_machine_actor_keys(128)
    assert all(k.startswith("job_critic.") for k in set(kop) - set(sd_op))
    assert all(k.startswith(("machine_critic.", "gat_layer.", "fcl_pooling.")) for k in set(km) - set(sd_m))
    sd_op = {**{k: torch.zeros(s) for k, s in kop.items()}, **sd_op}
    sd_m = {**{k: torch.zeros(s) for k, s in km.items()}, **sd_m}
    job = enc.EsaJobActor(sd_op, 6, 6, precision=precision)
    mch = enc.EsaMachineActor(sd_m, 6, precision=precision)
    out = val.greedy_validate(job, mch, inst)
    mine, csv, ref = out["final4"], g["csv14"], g["ref_cpu"]
    floor = int((ref == csv).all(axis=1).sum())
    same = int((mine == csv).all(axis=1).sum())
    same_ref = int((mine == ref).all(axis=1).sum())
    print("ESA %s: %d / 100 identical to CSV row 14, %d / 100 to the CPU reference (reference vs CSV: %d)"
          % (precision, same, same_ref, floor))
    assert same >= floor - min_same, (precision, same, floor)
    assert same_ref >= floor - min_same, (precision, same_ref)
    rel = abs(_objective(mine).mean() - _objective(csv).mean()) / _objective(csv).mean()
    assert rel < 5e-3, (precision, rel)


def _rollout_setup(J, M, E, B, mprec):
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
    d = ins.synthetic_instances(0, B, J, M, E, 41)
    w = ins.random_weights(0, B, 41)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    job = enc.EsaJobActor(enc.seeded_state_dict(enc.esa_job_actor_keys(128), 21), J, M)
    mch = enc.EsaMachineActor(enc.seeded_state_dict(enc.esa_machine_actor_keys(128), 22), M, precision=mprec)
    return env, job, mch, d, w


@pytest.mark.gpu
@pytest.mark.parametrize("J,M,E,B", [(6, 6, 2, 128), (10, 10, 3, 64)])
@pytest.mark.parametrize("mprec", ["fp32", "tf32"])
def test_esa_rollout_greedy_replays_on_the_oracle(J, M, E, B, mprec):
    from oracle.mtfjsp_oracle import OracleEnv

    ro_mod = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
    env, job, mch, d, w = _rollout_setup(J, M, E, B, mprec)
    ro = ro_mod.Rollout(env, job, mch, greedy=True)
    assert ro.job_v.shape == (B, 4)
    ro.begin_episode(w)
    ora = OracleEnv(B, J, M, E)
    ora.load(d["t"], d["p"], d["transT"], d["edge"])
    ora.scaler_init()
    ora.reset(w)
    for s in range(env.N):
        ro.step()
        assert not env.invalid.cpu().numpy().any()
        r5, s4, done, inv = ora.step(env.op.cpu().numpy(), env.mach.cpu().numpy())
        assert not inv.any()
        np.testing.assert_array_equal(env.reward5.cpu().numpy(), r5)
        np.testing.assert_array_equal(env.scaled4.cpu().numpy(), s4)
    assert env.done.cpu().numpy().all()
    np.testing.assert_array_equal(env.costs().cpu().numpy(), ora.costs())


@pytest.mark.gpu
@pytest.mark.parametrize("J,M,E,B", [(6, 6, 2, 256), (10, 10, 3, 64)])
def test_esa_sampled_rollout_graph_replay_equals_eager(J, M, E, B):
    """Sampled episode (one-launch selection, counter-based draws) with the tf32 ESA machine actor: CUDA-graph replays and
    eager steps with the same seed choose the same actions; every env finishes, no invalid action."""
    ro_mod = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.rollout")
    env, job, mch, d, w = _rollout_setup(J, M, E, B, "tf32")
    acts = {}
    for graph in (False, True):
        ro = ro_mod.Rollout(env, job, mch, greedy=False, use_cuda_graph=graph, seed=9)
        ro.begin_episode(w)
        seq = []
        for s in range(env.N):
            ro.step()
            seq.append(torch.stack((env.op, env.mach)).cpu().numpy())
            assert not env.invalid.any().item()
        assert env.done.all().item()
        acts[graph] = np.stack(seq)
    np.testing.assert_array_equal(acts[True], acts[False])
