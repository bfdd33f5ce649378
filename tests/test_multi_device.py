"""One thread drives device 0, then device 1, then device 0 again through every kind of launch the library sizes per
device: the tcgen05 layers that opt in to more than 48 KB of shared memory and size a persistent grid by the SM count
(the K = 128 TMA layer, both head forms, both trunk forms, the weight gradient), the hypervolume, and the env step, peek
and replay kernels.  Each launch must work on every device it meets, and give the same bits on each."""
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
pareto = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.pareto")

pytestmark = pytest.mark.gpu


def _env(J, M, E, B, dev):
    d = ins.synthetic_instances(0, B, J, M, E, seed=11)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, device="cuda:%d" % dev, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, seed=11))
    return env


def _outputs(dev):
    """Every output of the launches above on device `dev`, copied to the host."""
    out = {}
    with torch.cuda.device(dev):
        g = torch.Generator(device="cuda").manual_seed(7)
        rnd = lambda *shape: torch.randn(*shape, device="cuda", generator=g)
        H = 128
        W, b = rnd(H, H) / H ** 0.5, rnd(H) * 0.1
        x = rnd(5000, H)
        out["linear_tma"] = enc.linear_tf32(x, W, b)                      # K = 128, rows >= 4096: the TMA kernel
        gz = rnd(5000, H)
        out["wgrad_dW"], out["wgrad_db"] = enc.wgrad_tf32(gz, x)

        B, rpe = 8, 40
        hx = rnd(B * rpe, H)
        Wa, W1, b1, w2, b2 = rnd(H, H) / H ** 0.5, rnd(H, H) / H ** 0.5, rnd(H) * 0.2, rnd(H) / H ** 0.5, rnd(1)
        bias = rnd(B, H) * 0.5
        sc, sh = torch.rand(H, device="cuda", generator=g) + 0.5, rnd(H) * 0.3
        out["head"] = enc.head_tf32(hx, None, B, rpe, 0, sc, sh, Wa, bias, W1, b1, w2, b2)
        out["head_grouped"] = enc.head_tf32(hx, None, B, rpe, 0, sc.repeat(2, 1), sh.repeat(2, 1), Wa, bias, W1, b1, w2, b2)

        M = 6
        mch = enc.MachineActor(enc.seeded_state_dict(enc.machine_actor_keys(H), 12), M, precision="tf32")
        a = mch.w["gat_layer.a"]
        tw = (mch.w["m_fea_1_fcl.weight"], mch.w["m_fea_2_fcl.weight"], mch.w["gat_layer.W"].t().contiguous(),
              a[0, :H, 0].contiguous(), a[0, H:, 0].contiguous())
        f1, f2 = rnd(B * M, 6), rnd(B * M, 8)
        stats = torch.zeros(2 * H, dtype=torch.float64, device="cuda")
        out["trunk"] = enc.gat_trunk_tf32(f1, f2, *tw, stats=stats)
        out["trunk_stats"] = stats
        es = torch.zeros((B, 1, 2, H), dtype=torch.float64, device="cuda")
        out["trunk_grouped"] = enc.gat_trunk_tf32_grouped(f1, f2, *tw, es, M)
        out["trunk_grouped_stats"] = es

        rng = np.random.default_rng(3)
        obj = rng.uniform(0.0, 1.0, (3000, 3))
        out["hypervolume"] = pareto.hypervolume(obj, np.array([0, 1000, 3000]), np.full((2, 3), 1.1))

        env = _env(6, 6, 2, 256, dev)
        for s in range(env.N):
            env.policy_random(seed=5 + s)
            env.step_obs(env.op, env.mach)
            for k in ("reward5", "scaled4", "task_fea", "mach_fea", "candidate"):
                out["step_obs_%d_%s" % (s, k)] = getattr(env, k).clone()

        env = _env(10, 10, 3, 128, dev)
        acts = []
        for s in range(env.N):
            if s == env.N // 2:
                out["peek_r5"], out["peek_inv"] = env.peek_candidates()
            env.random_step(seed=9, env_offset=0)
            acts.append(torch.stack((env.op, env.mach), 1).clone())
        out["replay_final4"], out["replay_ret5"], out["replay_finv"] = env.replay(torch.stack(acts))
        out["costs"] = env.costs()
        torch.cuda.synchronize()
    return {k: v.cpu() for k, v in out.items()}


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_one_thread_alternating_devices():
    first = _outputs(0)
    for dev in (1, 0):
        again = _outputs(dev)
        assert again.keys() == first.keys()
        for k in first:
            np.testing.assert_array_equal(again[k].numpy(), first[k].numpy(), err_msg="%s on device %d" % (k, dev))
