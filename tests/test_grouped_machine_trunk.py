"""Per-group BatchNorm on the fused tcgen05 machine trunk (mtfjsp_enc_gat_trunk_tf32_grouped).

The grouped trunk runs the same per-machine arithmetic as mtfjsp_enc_gat_trunk_tf32 on env-aligned tiles of
(128 / M) * M machines and writes each env's column sums of the output and of its squares (row order, FP64, no
atomics).  Checked here, at every M from the edges of the size range: the statistics against FP64 sums of the output,
bitwise position independence, the output against the ungrouped kernel, and the tf32 machine actor with groups > 1
(per-group affines from these statistics applied by the pooling and the head) against the FP32 path with the same
groups."""
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
F = torch.nn.functional
pytestmark = pytest.mark.gpu

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")

SIZES = [(3, 2, 1), (6, 6, 2), (10, 10, 3), (6, 20, 5), (2, 64, 4)]   # M = 2, 6, 10, 20, 64


def _weights(mch):
    w, H = mch.w, mch.H
    a = w["gat_layer.a"]
    return (w["m_fea_1_fcl.weight"], w["m_fea_2_fcl.weight"], w["gat_layer.W"].t().contiguous(), a[0, :H, 0].contiguous(),
            a[0, H:, 0].contiguous())


def _features(J, M, E, B, seed=5, steps=2):
    """Machine features of real env states: B envs after `steps` random steps, the first candidate's machine rows."""
    d = ins.synthetic_instances(0, B, J, M, E, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed))
    env.obs(envm.MASK_ESA)
    for _ in range(steps):
        env.random_step(seed=3, env_offset=0)
        env.obs(envm.MASK_ESA)
    m1, mmask = env.mfea1(env.candidate[:, 0].contiguous())
    return env, m1.clone(), env.mach_fea.clone(), mmask.clone()


@pytest.mark.parametrize("size", SIZES)
def test_env_stats_and_position_independence(size):
    J, M, E = size
    B = 2 * (128 // M) + 3                     # more than two tiles, the last one partial
    env, f1, f2, _ = _features(J, M, E, B)
    mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(128), 12), M, precision="tf32")
    W = _weights(mch)

    def run(idx):
        idx = torch.tensor(idx, device="cuda")
        a = f1[idx].reshape(-1, 6).contiguous()
        b = f2[idx].reshape(-1, 8).contiguous()
        es = torch.full((len(idx), 1, 2, 128), float("nan"), dtype=torch.float64, device="cuda")
        return enc.gat_trunk_tf32_grouped(a, b, *W, es, M), es, a, b

    out, es, a, b = run(list(range(B)))
    z = out.double().view(B, M, 128)
    np.testing.assert_allclose(es[:, 0, 0].cpu().numpy(), z.sum(1).cpu().numpy(), rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(es[:, 0, 1].cpu().numpy(), (z ** 2).sum(1).cpu().numpy(), rtol=1e-12, atol=1e-9)
    ref = enc.gat_trunk_tf32(a, b, *W)        # the same per-machine arithmetic, batch-wide tiles
    np.testing.assert_allclose(out.cpu().numpy(), ref.cpu().numpy(), rtol=1e-6, atol=1e-6)

    for e in (0, B // 2, B - 1):
        o1, es1, _, _ = run([e])
        others = [i for i in range(B) if i != e]
        for order in ([e] + others[:3], others[:1] + [e] + others[1:4], others[: 128 // M] + [e], others + [e]):
            k = order.index(e)
            o, es, _, _ = run(order)
            assert torch.equal(es[k], es1[0]), (size, e, order)
            assert torch.equal(o.view(len(order), M, 128)[k], o1.view(M, 128)), (size, e, order)


class _FP32Trunk(enc.MachineActor):
    """The FP32 machine trunk up to (not including) its BatchNorm: the rows the statistics are taken over."""

    def pre_bn(self, f1, f2):
        w, B = self.w, f1.shape[0]
        h1 = F.linear(f1, w["m_fea_1_fcl.weight"]).reshape(B * self.M, self.H)
        h2 = F.linear(f2, w["m_fea_2_fcl.weight"]).reshape(B * self.M, self.H)
        h1, h2 = self._gat(h1, h2)
        h1, h2 = self._gat(F.elu(h1), F.elu(h2))
        h1, h2 = self._gat(F.elu(h1), F.elu(h2))
        return torch.stack((h1, h2), dim=1).mean(dim=-2)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("epg", [4, 16])
def test_grouped_machine_actor_matches_fp32(size, epg):
    """Per-group scale / shift against FP64 statistics of the kernel's own output, and against the FP32 path's; the
    machine actor's probabilities and values with groups = B / epg against the FP32 path with the same groups, within the
    tolerances the encoder tests give TF32 (rtol 3e-2, atol 5e-3)."""
    J, M, E = size
    B = 32
    G = B // epg
    env, f1, f2, mmask = _features(J, M, E, B, seed=9, steps=J * M // 2)
    sd = enc.seeded_state_dict(enc.machine_actor_keys(128), 12)
    m32, m16 = _FP32Trunk(sd, M, precision="fp32"), enc.MachineActor(sd, M, precision="tf32")
    h_o = torch.randn(B, 128, device="cuda", generator=torch.Generator("cuda").manual_seed(3)) / 3
    with torch.no_grad():
        p32, pool32, v32 = m32.forward(f1, f2, h_o, mmask, groups=G)
        p16, pool16, v16 = m16.forward(f1, f2, h_o, mmask, groups=G)
        hm = m32.pre_bn(f1, f2).double().view(G, epg * M, 128)
        buf, _ = m16.trunk(f1, f2, groups=G)
    sc, sh = m16._pending_m
    assert sc.shape == (G, 128)
    zg = buf.double().view(G, epg * M, 128)
    ksc = m16.w["bn.weight"].double() / torch.sqrt(zg.var(1, unbiased=False) + 1e-5)
    np.testing.assert_allclose(sc.double().cpu().numpy(), ksc.cpu().numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(sh.double().cpu().numpy(), (m16.w["bn.bias"].double() - zg.mean(1) * ksc).cpu().numpy(),
                               rtol=1e-5, atol=1e-5)
    mean, var = hm.mean(1), hm.var(1, unbiased=False)
    rsc = m32.w["bn.weight"].double() / torch.sqrt(var + 1e-5)
    rsh = m32.w["bn.bias"].double() - mean * rsc
    tol = dict(rtol=3e-2, atol=5e-3)
    # a column whose group variance is near zero (machines in identical states) has an ill-conditioned scale and shift
    # in either arithmetic; the normalised values there are near zero in both
    ok = (var > 1e-3).cpu().numpy()
    np.testing.assert_allclose(sc.double().cpu().numpy()[ok], rsc.cpu().numpy()[ok], **tol)
    np.testing.assert_allclose(sh.double().cpu().numpy()[ok], rsh.cpu().numpy()[ok], **tol)
    np.testing.assert_allclose(p16.cpu().numpy(), p32.cpu().numpy(), **tol)
    # the pooled embedding is a mean of normalised values: a TF32 operand error times the group's 1 / sigma, which reaches
    # about 30 for the small groups here, hence the wider absolute tolerance
    ok_env = np.repeat(ok, epg, axis=0)
    np.testing.assert_allclose(pool16.cpu().numpy()[ok_env], pool32.cpu().numpy()[ok_env], rtol=3e-2, atol=3e-2)
    np.testing.assert_allclose(v16.cpu().numpy(), v32.cpu().numpy(), **tol)


def test_grouped_trunk_rejects_bad_arguments():
    lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib").lib()
    x = torch.zeros(16, device="cuda")
    args = [x.data_ptr()] * 9
    assert lib.mtfjsp_enc_gat_trunk_tf32_grouped(*args, 4, 129, None) == -1     # M > 128
    assert lib.mtfjsp_enc_gat_trunk_tf32_grouped(*args, 0, 6, None) == -1       # B < 1
    assert lib.mtfjsp_enc_gat_trunk_tf32_grouped(*([None] + args[1:]), 4, 6, None) == -1
