"""Small invocations of every kernel family for compute-sanitizer (memcheck / racecheck / initcheck):
    compute-sanitizer --tool memcheck python profiles/sanitize_small.py [env|enc|all]"""
import importlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

what = sys.argv[1] if len(sys.argv) > 1 else "all"
pkg = importlib.import_module("e2e-mappo-for-mt-fjsp_b200")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")

if what in ("env", "all"):
    for (B, J, M, E) in ((37, 6, 6, 2), (21, 10, 10, 3), (5, 30, 20, 5), (9, 4, 5, 2), (11, 10, 6, 2), (7, 20, 6, 3), (9, 15, 10, 2),
                         (5, 20, 10, 5)):
        d = pkg.instances.synthetic_instances(0, B, J, M, E, 3)
        env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32)
        env.load(d["t"], d["p"], d["transT"], d["edge"])
        env.scaler_init()
        env.reset(pkg.instances.random_weights(0, B, 3))
        steps = min(J * M, 40)
        for s in range(steps):
            env.random_step(seed=1)
        act, rec = env.host_buffers()
        env.reset(pkg.instances.random_weights(0, B, 3))
        env.policy_random(seed=2)
        act[:, 0].copy_(env.op.cpu()); act[:, 1].copy_(env.mach.cpu())
        env.step_host_packed(act, rec)
        env.mfea1(env.op)
        env.dense_adj()
        env.costs()
        torch.cuda.synchronize()
        print("env ok", (B, J, M, E), int(env.invalid.sum()))

if what in ("enc", "all"):
    g = torch.Generator(device="cuda").manual_seed(1)
    for rows, K in ((300, 128), (77, 12), (1000, 64)):
        x = torch.randn(rows, K, device="cuda", generator=g)
        W = torch.randn(128, K, device="cuda", generator=g)
        b = torch.randn(128, device="cuda", generator=g)
        stats = torch.zeros(256, dtype=torch.float64, device="cuda")
        sc, sh = torch.rand(K, device="cuda") + 0.5, torch.randn(K, device="cuda")
        enc.linear_tf32(x, W, b)
        enc.linear_tf32(x, W, b, sc, sh, relu=True, stats=stats)
        enc.wgrad_tf32(torch.randn(rows, 128, device="cuda", generator=g), x)
    R = 50
    t = torch.randn(2 * R, 128, device="cuda")
    for mode in (0, 1, 2):
        enc.gat_attend(t, torch.randn(128, device="cuda"), torch.randn(128, device="cuda"), mode)
    # round-2 kernels: TMA layer (rows >= 4096), aggregation in the epilogue, one-launch head / trunk, selection
    rows = 4096 + 77
    x = torch.randn(rows, 128, device="cuda", generator=g)
    W = torch.randn(128, 128, device="cuda", generator=g) / 11.3
    b = torch.randn(128, device="cuda", generator=g)
    stats = torch.zeros(256, dtype=torch.float64, device="cuda")
    sc, sh = torch.rand(128, device="cuda") + 0.5, torch.randn(128, device="cuda")
    enc.linear_tf32(x, W, b)
    enc.linear_tf32(x, W, b, sc, sh, relu=True, stats=stats)
    for (Bq, N) in ((130, 36), (41, 100), (9, 128)):
        h = torch.randn(Bq, N, 128, device="cuda", generator=g)
        aw = torch.rand(Bq, N, 2, device="cuda", generator=g)
        aw[:, 0, 0] = 0.0
        asrc = torch.randint(-1, N, (Bq, N), device="cuda", generator=g, dtype=torch.int16)
        assert enc.aggregate_linear_tf32(h, aw, asrc, W, b, sc, sh, relu=True, stats=stats) is not None
    Bq = 300
    nodes = torch.randn(Bq, 36, 128, device="cuda", generator=g)
    cand = torch.randint(0, 36, (Bq, 6), device="cuda", generator=g, dtype=torch.int32)
    bias = torch.randn(Bq, 128, device="cuda", generator=g)
    enc.head_tf32(nodes, cand, Bq, 6, 36, sc, sh, W, bias, W, b, b, b[:1].contiguous())
    enc.head_tf32(nodes.reshape(-1, 128)[: Bq * 6].contiguous(), None, Bq, 6, 0, None, None, W, bias[:1].contiguous(), W, b, b,
                  b[:1].contiguous(), relu=False)
    enc.gat_trunk_tf32(torch.randn(777, 6, device="cuda"), torch.randn(777, 8, device="cuda"), torch.randn(128, 6, device="cuda"),
                       torch.randn(128, 8, device="cuda"), W, b, b, stats)
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    for R_ in (6, 20, 32):
        sco = torch.randn(501, R_, device="cuda", generator=g)
        msk = torch.rand(501, R_, device="cuda", generator=g) < 0.3
        enc.select(sco, msk, None, 1.0, False, (3, counter), 0)
        enc.select(sco, msk, torch.randint(0, 99, (501, R_), device="cuda", dtype=torch.int32), 10.0, True, None, 1)
    torch.cuda.synchronize()
    print("enc ok")
