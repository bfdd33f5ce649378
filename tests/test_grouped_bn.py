"""Per-instance BatchNorm groups on the tcgen05 job encoder, and batched sampled validation (best of K).

The grouped layers write per-env column statistics env_stats [B,P,2,128] (env-aligned tiles, each env summed in row
order), the grouped finalize turns them into one affine per group of envs, and every consumer applies the affine of its
env's group.  Checked here: the kernels against FP64 torch, bitwise position independence, the grouped tf32 job actor
against the FP32 per-instance path, batched greedy validation against the one-instance-per-batch run and the shipped
CSV rows, sampled rollouts replayed on the oracle, and the PPO-S row of the shipped CSV as a statistical target."""
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
val = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.validate")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")

SIZES = [(6, 6, 2), (10, 10, 3), (20, 6, 3), (15, 10, 2), (20, 10, 3), (30, 20, 5)]  # N = 36, 100, 120, 150, 200, 600


def _tf32(t):  # cvt.rna.tf32.f32 on the operands
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _shipped():
    g = np.load(os.path.join(GOLD, "policy_golden.npz"))
    pd = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    return g, {k: pd[k] for k in ("t", "p", "transT", "edge")}


class _GroupedAlways(enc.JobActor):
    """The grouped tf32 encoder even at one group (groups == 1 otherwise takes the batch-statistics kernels)."""

    def encode(self, task_fea, adj_w, adj_src, groups=1, adj_dst=None):
        return self._encode_tf32_grouped(task_fea.to(torch.float32), adj_w, adj_src, groups)


class _MachGroupedAlways(enc.MachineActor):
    """The machine actor's per-group BatchNorm path (gat_trunk_tf32, then mtfjsp_enc_bn_fwd) even at one group; with
    groups == 1 the tf32 machine actor otherwise folds batch-wide statistics into its head."""

    def trunk(self, machine_fea_1, machine_fea_2, groups=1):
        w, H, M = self.w, self.H, self.M
        B = machine_fea_1.shape[0]
        a = w["gat_layer.a"]
        buf = enc.gat_trunk_tf32(machine_fea_1.to(torch.float32).reshape(B * M, 6).contiguous(),
                                 machine_fea_2.to(torch.float32).reshape(B * M, 8).contiguous(), w["m_fea_1_fcl.weight"],
                                 w["m_fea_2_fcl.weight"], w["gat_layer.W"].t().contiguous(), a[0, :H, 0].contiguous(),
                                 a[0, H:, 0].contiguous())
        self._pending_m = None
        nodes = enc.bn_forward(buf, w["bn.weight"], w["bn.bias"], 1e-5, groups, False)[0].reshape(B, M, H)
        return nodes, nodes.mean(dim=1)


def _env(J, M, E, B, seed=77, steps=0):
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed))
    env.obs(envm.MASK_ESA)
    for _ in range(steps):
        env.random_step(seed=3, env_offset=0)
        env.obs(envm.MASK_ESA)
    return env, d


@pytest.mark.parametrize("N", [36, 100, 120, 150, 200, 600])
@pytest.mark.parametrize("epg", [1, 3, 16])
def test_grouped_kernels_against_fp64(N, epg):
    """linear (K = 4, 8, 12, 16 and K = 128 with a per-group affine), aggregation + layer, finalize, aggregation, pooling
    and the policy head against FP64 torch, B = 5 epg envs (not a multiple of the envs per tile for N = 36 with epg != 3)."""
    torch.manual_seed(N * 31 + epg)
    dev = torch.device("cuda")
    B = 5 * epg
    G = B // epg
    rows = B * N
    P = enc.env_stat_pieces(N)
    gid = torch.arange(rows, device=dev) // N // epg
    x12 = torch.randn(rows, 12, device=dev)
    W12 = torch.randn(128, 12, device=dev) / 4
    b = torch.randn(128, device=dev) / 4
    es = torch.full((B, P, 2, 128), float("nan"), dtype=torch.float64, device=dev)
    z = enc.linear_tf32_grouped(x12, N, W12, b, None, None, False, es)
    ref = _tf32(x12).double() @ _tf32(W12).double().T + b.double()
    np.testing.assert_allclose(z.double().cpu().numpy(), ref.cpu().numpy(), rtol=2e-5, atol=2e-5)
    for K in (4, 8, 16):  # the other widths the grouped first layer accepts
        xk, Wk = torch.randn(rows, K, device=dev), torch.randn(128, K, device=dev) / K ** 0.5
        esk = torch.full_like(es, float("nan"))
        zk = enc.linear_tf32_grouped(xk, N, Wk, b, None, None, False, esk)
        refk = _tf32(xk).double() @ _tf32(Wk).double().T + b.double()
        np.testing.assert_allclose(zk.double().cpu().numpy(), refk.cpu().numpy(), rtol=2e-5, atol=2e-5, err_msg="K=%d" % K)
        zd = zk.double().view(B, N, 128)
        np.testing.assert_allclose(esk[:, 0, 0].cpu().numpy(), zd[:, :128].sum(1).cpu().numpy(), rtol=1e-12, atol=1e-9)

    def check_stats(z, es):
        zd = z.double().view(B, N, 128)
        pad = torch.zeros((B, P * 128, 128), dtype=torch.float64, device=dev)
        pad[:, :N] = zd
        pieces = pad.view(B, P, 128, 128)
        np.testing.assert_allclose(es[:, :, 0].cpu().numpy(), pieces.sum(2).cpu().numpy(), rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(es[:, :, 1].cpu().numpy(), (pieces ** 2).sum(2).cpu().numpy(), rtol=1e-12, atol=1e-9)
        gamma, beta = torch.rand(128, device=dev) + 0.5, torch.randn(128, device=dev) / 5
        sc, sh = enc.bn_finalize_grouped(es, N, G, gamma, beta)
        zg = zd.view(G, epg * N, 128)
        mean, var = zg.mean(1), zg.var(1, unbiased=False)
        rsc = gamma.double() / torch.sqrt(var + 1e-5)
        np.testing.assert_allclose(sc.double().cpu().numpy(), rsc.cpu().numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(sh.double().cpu().numpy(), (beta.double() - mean * rsc).cpu().numpy(), rtol=1e-5, atol=1e-5)
        return sc, sh

    sc, sh = check_stats(z, es)
    W = torch.randn(128, 128, device=dev) / 11
    es2 = torch.full_like(es, float("nan"))
    z2 = enc.linear_tf32_grouped(z, N, W, b, sc, sh, True, es2)
    xin = torch.relu(z.double() * sc.double()[gid] + sh.double()[gid])
    # the kernel forms the affine with one FMA before rounding to TF32; torch rounds twice, so an operand can land one
    # TF32 step away (2^-11 relative) from the kernel's
    ref2 = _tf32(torch.relu(z * sc[gid] + sh[gid])).double() @ _tf32(W).double().T + b.double()
    np.testing.assert_allclose(z2.double().cpu().numpy(), ref2.cpu().numpy(), rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(z2.double().cpu().numpy(), (xin @ W.double().T + b.double()).cpu().numpy(), rtol=5e-3, atol=5e-3)
    check_stats(z2, es2)

    # aggregation with the per-group affine, its fused form with the layer, pooling: group by group against the
    # ungrouped kernels with that group's affine (the same per-row arithmetic, so the same bits)
    env, _ = _env(*{36: (6, 6, 2), 100: (10, 10, 3), 120: (20, 6, 3), 150: (15, 10, 2), 200: (20, 10, 3),
                    600: (30, 20, 5)}[N], B, steps=3)
    h = z.view(B, N, 128)
    agg = enc.aggregate(h, env.adj_w, env.adj_src, sc, sh, relu=True)
    pm = enc.graph_mean(h, sc, sh, relu=True)
    for g in range(G):
        s = slice(g * epg, (g + 1) * epg)
        assert torch.equal(agg[s], enc.aggregate(h[s], env.adj_w[s].contiguous(), env.adj_src[s].contiguous(), sc[g], sh[g], relu=True))
        assert torch.equal(pm[s], enc.graph_mean(h[s].contiguous(), sc[g], sh[g], relu=True))
    if N <= 128:
        es3 = torch.full_like(es, float("nan"))
        z3 = enc.aggregate_linear_tf32_grouped(h, env.adj_w, env.adj_src, W, b, sc, sh, True, es3)
        ref3 = _tf32(agg.reshape(rows, 128)).double() @ _tf32(W).double().T + b.double()
        np.testing.assert_allclose(z3.double().cpu().numpy(), ref3.cpu().numpy(), rtol=5e-3, atol=5e-3)
        check_stats(z3, es3)

    # policy head: candidate rows gathered, the affine of the row's group
    J = env.J
    cand = env.candidate.to(torch.int32).contiguous()
    Wa, W1 = torch.randn(128, 128, device=dev) / 11, torch.randn(128, 128, device=dev) / 11
    b1, w2, b2 = torch.randn(128, device=dev) / 5, torch.randn(128, device=dev) / 11, torch.randn(1, device=dev)
    bias = torch.randn(B, 128, device=dev) / 5
    out = enc.head_tf32(h, cand, B, J, N, sc, sh, Wa, bias, W1, b1, w2, b2)
    for g in range(G):
        s = slice(g * epg, (g + 1) * epg)
        one = enc.head_tf32(h[s].contiguous(), cand[s].contiguous(), epg, J, N, sc[g].contiguous(), sh[g].contiguous(), Wa,
                            bias[s].contiguous(), W1, b1, w2, b2)
        assert torch.equal(out[s], one)


@pytest.mark.parametrize("size", [(6, 6, 2), (15, 10, 2)])
def test_position_independence_is_bitwise(size):
    """An env's statistics and job-actor probabilities are the same bits alone and at several batch positions (tile
    offsets 0 / 36 / 72 at N = 36; multi-piece envs at N = 150)."""
    J, M, E = size
    N = J * M
    B = 11
    env, _ = _env(J, M, E, B, steps=2)
    sdj = enc.seeded_state_dict(enc.job_actor_keys(128), 21)
    job = _GroupedAlways(sdj, J, M, precision="tf32")
    W12 = torch.randn(128, 12, device="cuda", generator=torch.Generator("cuda").manual_seed(1)) / 4

    def run(idx):
        idx = torch.tensor(idx, device="cuda")
        tf, aw, asrc = env.task_fea[idx].contiguous(), env.adj_w[idx].contiguous(), env.adj_src[idx].contiguous()
        es = torch.empty((len(idx), enc.env_stat_pieces(N), 2, 128), dtype=torch.float64, device="cuda")
        enc.linear_tf32_grouped(tf.reshape(-1, 12), N, W12, None, None, None, False, es)
        with torch.no_grad():
            p, _, _ = job.evaluate(tf, aw, asrc, env.candidate[idx].contiguous(), None, env.job_mask[idx].contiguous(),
                                   groups=len(idx))
        return es, p

    for e in (0, 4, 10):
        es1, p1 = run([e])
        for order in ([e, 1, 2, 3], [1, e, 2, 3, 5], [1, 2, e, 3], [3, 5, 6, 7, 8, 9, 2, e], list(range(B))):
            k = order.index(e)
            es, p = run(order)
            assert torch.equal(es[k], es1[0]), (e, order)
            assert torch.equal(p[k], p1[0]), (e, order)


@pytest.mark.parametrize("size", SIZES)
def test_grouped_tf32_matches_fp32_per_instance(size):
    """First-step job probabilities of the grouped tf32 job actor against the FP32 path with per-instance groups."""
    J, M, E = size
    B = 9
    env, _ = _env(J, M, E, B, steps=1)
    sdj = enc.seeded_state_dict(enc.job_actor_keys(128), 21)
    with torch.no_grad():
        p = {prec: enc.JobActor(sdj, J, M, precision=prec).evaluate(env.task_fea, env.adj_w, env.adj_src, env.candidate, None,
                                                                    env.job_mask, groups=B)[0] for prec in ("fp32", "tf32")}
    np.testing.assert_allclose(p["tf32"].cpu().numpy(), p["fp32"].cpu().numpy(), rtol=5e-2, atol=5e-3)


@pytest.mark.parametrize("tag,row", [("iotj", "csv15"), ("n12800", "csv17")])
def test_batched_greedy_validation_equals_one_instance_batches(tag, row):
    g, inst = _shipped()
    sd_op, sd_m = val.load_actor_state_dicts(g, tag)
    batched = val.greedy_validate(enc.JobActor(sd_op, 6, 6, precision="tf32"), enc.MachineActor(sd_m, 6, precision="tf32"), inst,
                                  chunk=100, return_actions=True)
    single = val.greedy_validate(_GroupedAlways(sd_op, 6, 6, precision="tf32"), _MachGroupedAlways(sd_m, 6, precision="tf32"),
                                 inst, chunk=1, return_actions=True)
    np.testing.assert_array_equal(batched["final4"], single["final4"])
    np.testing.assert_array_equal(batched["actions"], single["actions"])
    same = int((batched["final4"] == g[row]).all(axis=1).sum())
    print("grouped tf32 batch of 100, %s: %d / 100 instances equal CSV %s" % (tag, same, row))
    assert same >= 90, (tag, same)


def _replay(inst, actions, idx, final4):
    from oracle.mtfjsp_oracle import OracleEnv

    n = len(idx)
    ora = OracleEnv(n, 6, 6, 2, left_shift=True)
    ora.load(*(np.asarray(inst[k])[idx] for k in ("t", "p", "transT", "edge")))
    ora.scaler_init()
    ora.reset(np.tile([0.4, 0.4, 0.2], (n, 1)))
    for step in range(actions.shape[0]):
        _, _, _, inv = ora.step(actions[step, :, 0], actions[step, :, 1])
        assert not inv.any()
    np.testing.assert_array_equal(ora.costs(), final4)


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_sampled_rollouts_replay_on_the_oracle(precision):
    g, inst = _shipped()
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    job, mch = enc.JobActor(sd_op, 6, 6, precision=precision), enc.MachineActor(sd_m, 6, precision=precision)
    K, S = 8, 100
    out = val.sampled_validate(job, mch, inst, samples=K, seed=11, max_envs=300, return_actions=True)  # 3 chunks
    assert out["final4"].shape == (K, S, 4) and out["objective"].shape == (K, S)
    assert out["actions"].shape == (36, K, S, 2)
    idx = np.tile(np.arange(S), K)
    _replay(inst, out["actions"].reshape(36, K * S, 2), idx, out["final4"].reshape(K * S, 4))
    best = out["objective"].argmin(axis=0)
    np.testing.assert_array_equal(out["best_index"], best)
    np.testing.assert_array_equal(out["best_objective"], out["objective"].min(axis=0))
    np.testing.assert_array_equal(out["best_final4"], out["final4"][best, np.arange(S)])
    _replay(inst, out["best_actions"], np.arange(S), out["best_final4"])
    again = val.sampled_validate(job, mch, inst, samples=K, seed=11, max_envs=300)
    np.testing.assert_array_equal(again["final4"], out["final4"])
    assert len(np.unique(out["objective"], axis=0)) > 1  # the K samples differ


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_sampled_iotj_matches_the_ppo_s_row(precision):
    """PPO-S (CSV row 16: the shipped iotj checkpoint with greedy=False, one sample per instance) against K = 256 samples
    per instance: the row's mean objective within 4 standard errors of the mean of the per-instance sample means, and the
    randomized PIT of each CSV value within its instance's samples uniform (Kolmogorov-Smirnov, p > 1e-3)."""
    from scipy import stats

    g, inst = _shipped()
    s16 = np.load(os.path.join(GOLD, "sampled_golden.npz"))["csv16"]
    sd_op, sd_m = val.load_actor_state_dicts(g, "iotj")
    job, mch = enc.JobActor(sd_op, 6, 6, precision=precision), enc.MachineActor(sd_m, 6, precision=precision)
    out = val.sampled_validate(job, mch, inst, samples=256, seed=2024)
    obj = out["objective"]                                       # [K, 100]
    csv = 0.4 * s16[:, 0] + 0.4 * (s16[:, 1] + s16[:, 3]) + 0.2 * s16[:, 2]
    se = np.sqrt(obj.var(axis=0, ddof=1).sum()) / obj.shape[1]
    z = (csv.mean() - obj.mean(axis=0).mean()) / se
    rs = np.random.RandomState(7)
    below, tie = (obj < csv).sum(axis=0), (obj == csv).sum(axis=0)
    pit = (below + rs.uniform(size=tie.shape) * (tie + 1)) / (obj.shape[0] + 1)
    p = stats.kstest(pit, "uniform").pvalue
    print("PPO-S %s: csv mean %.2f, sampled mean %.2f, z = %.2f, KS p = %.3g" % (precision, csv.mean(), obj.mean(), z, p))
    assert abs(z) < 4, z
    assert p > 1e-3, p
