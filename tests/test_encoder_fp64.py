"""The tcgen05 inference encoder against FP64 references computed from each kernel's inputs.

No reference here is the output of another project kernel.  Where a kernel rounds an operand, the reference rounds it
the same way: GEMM operands to TF32 as `cvt.rna.tf32.f32` does (`_tf32`), and the folded BatchNorm of the producing
layer as the kernels' one FP32 fused multiply-add, float32(x * scale + shift) formed in FP64, then ReLU (`_affine`).

1. The consumers of the folded BatchNorm: the aggregation (all three neighbourhood members, real mid-episode and
   last-step adjacency at every specialised size and one without a specialisation), the graph mean, the fused
   aggregation + layer, and the policy head gathering candidate rows above 128 nodes per env.
2. The whole TF32 job actor against the FP64 restatement of tests/test_update_gradients.py run as a TF32 shadow (its
   operands rounded where the tcgen05 path rounds them, its order of aggregation and product, its split head).
3. The C ABI refuses misaligned operands and out-of-range arguments on the host, before anything is launched.
"""
import ctypes as C
import functools
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
enc = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.encoder")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
_lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

U = 2.0 ** -24  # FP32 unit roundoff
# the seven sizes with a specialised env kernel (N = 36 ... 600) and one without (J13M11, N = 143)
SIZES = [(6, 6, 2), (10, 6, 2), (10, 10, 3), (20, 6, 3), (15, 10, 2), (20, 10, 3), (30, 20, 5), (13, 11, 3)]
sid = lambda s: "J%dM%dE%d" % s


def _tf32(t):  # cvt.rna.tf32.f32: round to nearest, ties away, on the 13 dropped mantissa bits
    i = t.float().contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _affine(h, sc, sh, relu):
    """The folded BatchNorm as the kernels apply it: one FP32 FMA (exact product and sum in FP64, one rounding)."""
    x = (h.double() * sc.double() + sh.double()).float()
    return torch.relu(x) if relu else x


def _bn_params(C, gen, G=None):
    shape = (C,) if G is None else (G, C)
    sign = torch.where(torch.rand(shape, device="cuda", generator=gen) < 0.2, -1.0, 1.0)
    sc = ((torch.rand(shape, device="cuda", generator=gen) + 0.25) * sign).contiguous()
    return sc, (torch.randn(shape, device="cuda", generator=gen) * 0.5).contiguous()


@functools.lru_cache(maxsize=None)
def _episode(J, M, E, B):
    """Observations of B envs under the random policy after N // 2 steps and after N - 1 (the last op left): machine arcs,
    coincident job / machine arcs and removed arcs all occur.  A = the env's dense adjacency adj[dst, src], diagonal 1."""
    N = J * M
    d = ins.synthetic_instances(0, B, J, M, E, 5)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, obs_dtype=torch.float32, mask_mode=envm.MASK_FINISHED)  # every open job a choice
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ins.random_weights(0, B, 5))
    env.obs()
    out = {}
    for s in range(1, N):
        env.random_step(seed=9)
        if s in (N // 2, N - 1):
            out["mid" if s == N // 2 else "last"] = {
                "task_fea": env.task_fea.clone(), "adj_w": env.adj_w.clone(), "adj_src": env.adj_src.clone(),
                "candidate": env.candidate.clone(), "job_mask": env.job_mask.clone(), "A": env.dense_adj(torch.float64)}
    torch.cuda.synchronize()
    return out


def _synthetic_adjacency(B, N, M, gen):
    """Random ELL rows: job arcs dropped at every M-th row and at random, machine predecessors anywhere in the env
    (also v - 1, beside a job arc), weights in [0.5, 1.5)."""
    adj_w = torch.rand(B, N, 2, device="cuda", generator=gen) + 0.5
    adj_w[:, ::M, 0] = 0.0
    adj_w[:, 0, 0] = 0.0
    adj_src = torch.randint(-1, N, (B, N), device="cuda", generator=gen, dtype=torch.int16)
    adj_w[..., 1] = torch.where(adj_src >= 0, adj_w[..., 1], torch.zeros_like(adj_w[..., 1]))
    drop = torch.rand(B, N, device="cuda", generator=gen) < 0.3
    adj_w[..., 0] = torch.where(drop, torch.zeros_like(adj_w[..., 0]), adj_w[..., 0])
    return adj_w.contiguous(), adj_src.contiguous()


def _ell_mean(y, adj_w, adj_src):
    """(y[v] + w_job y[v-1] + w_mach y[src]) / (number of members), FP64, straight from the ELL rows."""
    B, N, _ = y.shape
    wj, wm = adj_w[..., 0].double().unsqueeze(-1), adj_w[..., 1].double().unsqueeze(-1)
    hj, hm = (adj_w[..., 0] != 0).unsqueeze(-1), (adj_src >= 0).unsqueeze(-1)
    prev = torch.cat((torch.zeros_like(y[:, :1]), y[:, :-1]), dim=1)
    src = torch.gather(y, 1, adj_src.long().clamp(min=0).unsqueeze(-1).expand_as(y))
    n = 1.0 + hj.double() + hm.double()
    return (y + torch.where(hj, wj * prev, 0.0) + torch.where(hm, wm * src, 0.0)) / n, n


# ---- 1. the folded-BatchNorm consumers --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=sid)
def test_aggregate_applies_the_folded_batchnorm_to_every_member(size, relu):
    """aggregate / aggregate_grouped with the input affine on real adjacency (mid-episode and last step) against the
    dense FP64 product of the env's adjacency with the post-affine rows, divided by the in-degree: within 3 FP32 ulp of
    the magnitude sum |A| |x| / deg (the bound of test_encoder.py).  An affine that misses the job or the machine
    predecessor, or a ReLU taken before it, is off by the size of the rows."""
    J, M, E = size
    N, B, epg = J * M, 8, 2
    gen = torch.Generator(device="cuda").manual_seed(N + relu)
    for state, st in _episode(J, M, E, B).items():
        A = st["A"]
        deg = (A != 0).sum(-1, keepdim=True).double()
        assert float(deg.max()) == 3.0 and float(deg.min()) < 3.0, (state, deg.unique())
        for Cc in (20, 128):  # C / 4 = 5 takes the division form of the row index, 32 the shift
            h = (torch.randn(B, N, Cc, device="cuda", generator=gen) * 1.5 + 0.3).contiguous()
            for grouped in (False, True):
                sc, sh = _bn_params(Cc, gen, B // epg if grouped else None)
                gid = torch.arange(B, device="cuda") // epg
                x = _affine(h, sc[gid].unsqueeze(1), sh[gid].unsqueeze(1), relu) if grouped else _affine(h, sc, sh, relu)
                out = enc.aggregate(h, st["adj_w"], st["adj_src"], sc, sh, relu=relu)
                ref = torch.bmm(A, x.double()) / deg
                bound = 3 * U * torch.bmm(A.abs(), x.double().abs()) / deg + 1e-30
                r = float(((out.double() - ref).abs() / bound).max())
                assert r <= 1.0, (state, Cc, grouped, r)


@pytest.mark.gpu
@pytest.mark.parametrize("relu", [True, False])
def test_aggregate_with_the_affine_on_synthetic_adjacency(relu):
    """Synthetic ELL rows (every member count, machine predecessor v - 1 beside a job arc) at N = 100 and 143, against
    the mean formed from the ELL rows in FP64; same bound."""
    gen = torch.Generator(device="cuda").manual_seed(3 + relu)
    for N, M in ((100, 10), (143, 11)):
        B = 37
        adj_w, adj_src = _synthetic_adjacency(B, N, M, gen)
        h = torch.randn(B, N, 128, device="cuda", generator=gen)
        sc, sh = _bn_params(128, gen)
        x = _affine(h, sc, sh, relu).double()
        out = enc.aggregate(h, adj_w, adj_src, sc, sh, relu=relu)
        ref, n = _ell_mean(x, adj_w, adj_src)
        assert {1.0, 2.0, 3.0} <= set(n.unique().tolist())
        bound = 3 * U * _ell_mean(x.abs(), adj_w.abs(), adj_src)[0] + 1e-30
        r = float(((out.double() - ref).abs() / bound).max())
        assert r <= 1.0, (N, r)


@pytest.mark.gpu
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("N", [36, 143, 600])
def test_graph_mean_with_the_folded_batchnorm(N, relu):
    """graph_mean / graph_mean_grouped with the input affine against the FP64 mean of the post-affine rows.  The kernel
    multiplies each row by the FP32 value 1/N and adds the rows in order: with u = 2^-24, that is at most (N + 1) u sum|x| / N
    (N - 1 additions, one rounding of each product, one of 1/N), plus u sum|h sc| / N should the affine's product be
    rounded before the shift is added."""
    gen = torch.Generator(device="cuda").manual_seed(N * 2 + relu)
    B = 32
    for Cc in (20, 128):
        h = (torch.randn(B, N, Cc, device="cuda", generator=gen) + 0.2).contiguous()
        for epg in (None, 4):
            sc, sh = _bn_params(Cc, gen, None if epg is None else B // epg)
            gsc = sc if epg is None else sc.repeat_interleave(epg, 0).unsqueeze(1)
            gsh = sh if epg is None else sh.repeat_interleave(epg, 0).unsqueeze(1)
            x = _affine(h, gsc, gsh, relu).double()
            out = enc.graph_mean(h, sc, sh, relu=relu)
            ref = x.mean(dim=1)
            bound = ((N + 1) * x.abs().sum(1) + (h.double() * gsc.double()).abs().sum(1)) * U * 1.01 / N + 1e-30
            r = float(((out.double() - ref).abs() / bound).max())
            assert r <= 1.0, (Cc, epg, r)


@pytest.mark.gpu
@pytest.mark.parametrize("wave", ["partial", "several"])
@pytest.mark.parametrize("N", [36, 60, 100, 120, 128])
def test_fused_aggregation_and_layer_against_fp64(N, wave):
    """aggregate_linear_tf32 against FP64 from h: the TF32-rounded rows relu(affine(h)), their product with the TF32-
    rounded weights, then the weighted mean of the PRODUCT rows (the kernel's order, DESIGN.md section 6) plus the bias.
    What is left is FP32 accumulation: the tolerance of test_tcgen05_linear_matches_fp32_matmul.  Batches of fewer tiles
    than one wave of 148 CTAs, and of more than two waves."""
    gen = torch.Generator(device="cuda").manual_seed(N * 5 + len(wave))
    ept = 128 // N  # whole envs per tile
    B = ept * 37 + 1 if wave == "partial" else ept * 148 * 2 + ept + 1
    M = {36: 6, 60: 6, 100: 10, 120: 6, 128: 8}[N]
    adj_w, adj_src = _synthetic_adjacency(B, N, M, gen)
    h = torch.randn(B, N, 128, device="cuda", generator=gen)
    W = torch.randn(128, 128, device="cuda", generator=gen) / 128 ** 0.5
    b = torch.randn(128, device="cuda", generator=gen)
    for relu in (True, False):
        sc, sh = _bn_params(128, gen)
        z = enc.aggregate_linear_tf32(h, adj_w, adj_src, W, b, sc, sh, relu=relu)
        assert z is not None
        y = (_tf32(_affine(h, sc, sh, relu)).double() @ _tf32(W).double().T)
        ref = _ell_mean(y, adj_w, adj_src)[0].reshape(B * N, 128) + b.double()
        np.testing.assert_allclose(z.double().cpu().numpy(), ref.cpu().numpy(), rtol=2e-5, atol=3e-5, err_msg="relu=%s" % relu)


@pytest.mark.gpu
@pytest.mark.parametrize("groups", [None, 1, 16], ids=["ungrouped", "epg1", "epg16"])
@pytest.mark.parametrize("bias_rows", ["B", "1"])
@pytest.mark.parametrize("nodes", [150, 200, 600])
def test_policy_head_gathers_candidates_above_128_nodes(nodes, bias_rows, groups):
    """head_tf32 gathering candidate rows from envs of 150, 200 and 600 nodes (J15M10, J20M10, J30M20; candidates
    anywhere in the env), ungrouped and with one affine per group of 1 or 16 envs, against the FP64 chain of
    test_fused_policy_head_matches_the_separate_launches on TF32-rounded operands."""
    gen = torch.Generator(device="cuda").manual_seed(nodes + len(bias_rows) + (groups or 0))
    H, rpe, B = 128, {150: 15, 200: 20, 600: 30}[nodes], 48
    x = torch.randn(B, nodes, H, device="cuda", generator=gen)
    cand = torch.randint(0, nodes, (B, rpe), device="cuda", generator=gen, dtype=torch.int32)
    assert bool((cand >= 128).any())
    sc, sh = _bn_params(H, gen, None if groups is None else B // groups)
    gsc = sc if groups is None else sc.repeat_interleave(groups, 0).unsqueeze(1)
    gsh = sh if groups is None else sh.repeat_interleave(groups, 0).unsqueeze(1)
    per_row = torch.gather(_affine(x, gsc, gsh, True), 1, cand.long().unsqueeze(-1).expand(-1, rpe, H)).reshape(B * rpe, H)
    Wa = torch.randn(H, H, device="cuda", generator=gen) / H ** 0.5
    W1 = torch.randn(H, H, device="cuda", generator=gen) / H ** 0.5
    b1 = torch.randn(H, device="cuda", generator=gen) * 0.2
    w2 = torch.randn(H, device="cuda", generator=gen) / H ** 0.5
    b2 = torch.randn(1, device="cuda", generator=gen)
    bias = torch.randn(B if bias_rows == "B" else 1, H, device="cuda", generator=gen) * 0.5
    out = enc.head_tf32(x, cand, B, rpe, nodes, sc, sh, Wa, bias, W1, b1, w2, b2)
    brow = bias.double().repeat_interleave(rpe, dim=0) if bias_rows == "B" else bias.double()
    z = torch.tanh((_tf32(per_row).double() @ _tf32(Wa).double().T + brow).float())
    z = torch.tanh((_tf32(z).double() @ _tf32(W1).double().T + b1.double()).float())
    ref = (z.double() @ w2.double() + b2.double()).view(B, rpe)
    np.testing.assert_allclose(out.double().cpu().numpy(), ref.cpu().numpy(), rtol=2e-4, atol=2e-4)


# ---- 2. the whole TF32 job actor against the TF32 shadow of the FP64 restatement ---------------------------------------
def _record(monkeypatch):
    """Wraps the encoder module's layer and BatchNorm-finalize entry points so that the outputs of one forward can be
    read layer by layer: (layer outputs in call order, (scale, shift) in call order)."""
    layers, affines = [], []

    def wrap(fn, into):
        def f(*a, **k):
            out = fn(*a, **k)
            if out is not None:
                into.append(out)
            return out
        return f

    for name in ("linear_tf32", "aggregate_linear_tf32", "linear_tf32_grouped", "aggregate_linear_tf32_grouped"):
        monkeypatch.setattr(enc, name, wrap(getattr(enc, name), layers))
    for name in ("bn_finalize", "bn_finalize_grouped"):
        monkeypatch.setattr(enc, name, wrap(getattr(enc, name), affines))
    return layers, affines


def _bn_affine64(z, w, b, groups):
    """scale, shift [G,C] of BatchNorm1d with batch statistics per group, FP64."""
    zs = z.reshape(groups, -1, z.shape[-1])
    var, mean = torch.var_mean(zs, dim=1, unbiased=False)
    sc = w / torch.sqrt(var + 1e-5)
    return sc, b - mean * sc


LAYERS = ["l%d.%d" % (l, i) for l in (0, 1) for i in (0, 1, 2)]
BN_NAMES = ["encoder.feature_extract.mlps.%d.batch_norms.%d." % (l, i) if i < 2 else "encoder.feature_extract.batch_norms.%d." % l
            for l in (0, 1) for i in (0, 1, 2)]
# Worst errors over all 40 cases (NVIDIA B200, 1000 W power limit) -> tolerance, at most 10 x the observed worst and at
# least 10 x tighter than the 5e-2 / 3e-2 of the tf32 parity tests.  Layer by layer (each layer from the device's layer
# before): node rows 1.7e-5 -> 1.5e-4, last affine 2.7e-7 -> 2.5e-6, pooled 3.1e-7 -> 3e-6, probabilities 5.0e-6 ->
# 5e-5, value 1.4e-4 -> 1.4e-3; Linear outputs l0.0 7.8e-7, l0.1 1.4e-5, l0.2 1.2e-5, l1.0 2.1e-5, l1.1 1.5e-5, l1.2
# 1.7e-5; affines <= 3.2e-7.  Free-running: node rows 4.6e-4 -> 4.5e-3, last affine 2.6e-3 -> 5e-3, pooled 2.6e-4 ->
# 2.5e-3, probabilities 6.3e-5 -> 6e-4, value 4.8e-4 -> 3e-3.
SHADOW_TOL = {"nodes": 1.5e-4, "affine": 2.5e-6, "pooled": 3e-6, "prob": 5e-5, "value": 1.4e-3,
              "layer l0.0": 7e-6, "layer l0.1": 1.3e-4, "layer l0.2": 1.1e-4, "layer l1.0": 2e-4, "layer l1.1": 1.4e-4,
              "layer l1.2": 1.5e-4, "free nodes": 4.5e-3, "free affine": 5e-3, "free pooled": 2.5e-3, "free prob": 6e-4,
              "free value": 3e-3}
SHADOW_TOL.update({"bn " + n: 3e-6 for n in LAYERS})


def _shadow_configs():
    out = []
    for size in SIZES:
        N = size[0] * size[1]
        small = max(1, min(16, 4095 // N))                 # every K = 128 layer below 4,096 rows: cp.async operands
        large = 16 * max(2, -(-4097 // (16 * N)))          # above: TMA operands
        out += [(size, small, 1), (size, small, small), (size, large, 1), (size, large, large), (size, large, large // 16)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("size,B,groups", _shadow_configs(), ids=lambda v: sid(v) if isinstance(v, tuple) else str(v))
def test_tf32_job_actor_against_the_fp64_tf32_shadow(size, B, groups, monkeypatch):
    """JobActor(precision="tf32") against f64_job_evaluate with the TF32 rounding hook, mid-episode and at the last step,
    with batch-wide BatchNorm (groups = 1) and per-group (groups = B, B / 16).

    Layer by layer (`feed`): each Linear of the shadow starts from the device's output of the layer before, so every
    layer -- its BatchNorm affine, TF32 operands, product, aggregation order -- is checked on its own, and the outputs
    (the encoder's node rows before the last BatchNorm, that BatchNorm's affine, pooled, the job probabilities, the job
    value) are checked from the device's last layer.  Errors: activations and pooled |d - s| / |s| in 2-norms over the
    tensor, affines relative to their largest entry, probabilities and values absolute.

    Free-running ("free": the shadow never sees a device value), the same five outputs.  The two runs agree to FP32
    accumulation noise only while they round an operand to the same TF32 value; each BatchNorm rescales what the layer
    before left, more operands land on the other side of a TF32 rounding boundary (a 2^-11 relative step), and the
    difference grows by about 3-4 x per Linear (2-norm 7.8e-7 after the first, 4.6e-4 after the sixth; single entries
    reach a few percent of the RMS where an operand far out in its column is rounded one TF32 step apart).  So the tight
    bounds are the layer-by-layer ones, and the free-running outputs are held to the measured growth.  Measured errors
    and tolerances: SHADOW_TOL."""
    tug = importlib.import_module("tests.test_update_gradients")
    J, M, E = size
    sd = enc.seeded_state_dict(enc.job_actor_keys(128), 21)
    job = enc.JobActor(sd, J, M, precision="tf32")
    w64 = {k: v.detach().to("cuda") for k, v in tug.f64_params("job", 128, sd=sd).items()}
    rnd = lambda t: _tf32(t).double()
    worst, lines = {}, []

    def err(name, got, ref, mode):
        if mode == "norm":  # |d - s| / |s|, 2-norms over the whole tensor
            e = float((got.double() - ref).norm() / ref.norm().clamp(min=1e-30))
        else:
            e = float((got.double() - ref).abs().max() / (ref.abs().max().clamp(min=1e-30) if mode == "max" else 1.0))
        worst[name] = max(worst.get(name, 0.0), e)
        return e

    def bn_err(name, affine, z, k):
        rsc, rsh = _bn_affine64(z, w64[BN_NAMES[k] + "weight"], w64[BN_NAMES[k] + "bias"], groups)
        return max(err(name, affine[0].reshape(rsc.shape), rsc, "max"), err(name, affine[1].reshape(rsh.shape), rsh, "max"))

    for state, st in _episode(J, M, E, B).items():
        layers, affines = _record(monkeypatch)
        with torch.no_grad():
            prob, pooled, jv = job.evaluate(st["task_fea"], st["adj_w"], st["adj_src"], st["candidate"], None, st["job_mask"],
                                            groups=groups)
        monkeypatch.undo()
        torch.cuda.synchronize()
        assert int((st["job_mask"] == 0).sum(1).max()) > 1 or state == "last"
        for mode in ("free", "fed"):
            trace, pre = [], "" if mode == "fed" else "free "
            with torch.no_grad():
                rprob, rpooled, rjv = tug.f64_job_evaluate(w64, st["task_fea"], st["A"], st["candidate"], None, st["job_mask"], groups,
                                                           rnd=rnd, trace=trace, feed=layers[:6] if mode == "fed" else None)
            per_layer = ["%s %.1e bn %.1e" % (n, err(pre + "layer " + n, layers[k], trace[k], "norm"),
                                              bn_err(pre + "bn " + n, affines[k], layers[k] if mode == "fed" else trace[k], k))
                         for k, n in enumerate(LAYERS)]
            out = {"nodes": err(pre + "nodes", layers[5], trace[5], "norm"),
                   "affine": bn_err(pre + "affine", affines[5], layers[5] if mode == "fed" else trace[5], 5),
                   "pooled": err(pre + "pooled", pooled, rpooled, "norm"),
                   "prob": err(pre + "prob", prob, rprob, "abs"),
                   "value": err(pre + "value", jv, rjv, "abs")}
            lines.append("%s %s: %s | %s" % (state, mode, ", ".join("%s %.1e" % kv for kv in out.items()), ", ".join(per_layer)))
    msg = "%s B=%d groups=%d\n%s\nworst: %s" % (sid(size), B, groups, "\n".join(lines),
                                                ", ".join("%s %.2e" % kv for kv in sorted(worst.items())))
    print(msg)
    bad = {k: worst[k] for k in SHADOW_TOL if worst[k] > SHADOW_TOL[k]}
    assert not bad, (bad, msg)


# ---- 3. the C ABI: misaligned operands and out-of-range arguments ------------------------------------------------------
# every encoder entry point that moves operands 16 (or 8) bytes at a time: argument list with named buffers, the names
# that must be 16-byte aligned, those that must be 8-byte aligned.  B = 2 envs of N = 36 rows, C = 128.
_ABI = {
    "mtfjsp_enc_aggregate": ("h adj_w adj_src out 2 36 128 sc sh 1 S", "h out sc sh", "adj_w"),
    "mtfjsp_enc_aggregate_grouped": ("h adj_w adj_src out 2 36 128 sc sh 1 1 S", "h out sc sh", "adj_w"),
    "mtfjsp_enc_aggregate_bwd": ("h adj_w adj_src adj_dst out 2 36 128 S", "h out", "adj_w"),
    "mtfjsp_enc_bn_fwd": ("h w b 1e-5 2 36 128 1 out mean rstd ws S", "h w b out mean rstd", "ws"),
    "mtfjsp_enc_bn_bwd": ("h g w b mean rstd 2 36 128 1 out ws S", "h g w b mean rstd out", "ws"),
    "mtfjsp_enc_gat_attend": ("h a_src a_dst out 72 1 S", "h a_src a_dst out", ""),
    "mtfjsp_enc_gat_attend_bwd": ("h a_src a_dst g out parts 72 1 S", "h a_src a_dst g out parts", ""),
    "mtfjsp_enc_linear_tf32": ("h 72 128 W bias sc sh 1 out ws S", "h W out", "ws"),
    "mtfjsp_enc_aggregate_linear_tf32": ("h 2 36 adj_w adj_src W bias sc sh 1 out ws S", "h W out", "adj_w ws"),
    "mtfjsp_enc_linear_tf32_grouped": ("h 2 36 128 W bias sc sh 1 1 out ws S", "h W out sc sh", "ws"),
    "mtfjsp_enc_aggregate_linear_tf32_grouped": ("h 2 36 adj_w adj_src W bias sc sh 1 1 out ws S", "h W out sc sh", "adj_w ws"),
    "mtfjsp_enc_head_tf32": ("h cand 2 6 36 sc sh 1 W bias 2 W1 b1 w2 b2 out S", "h W bias W1", ""),
    "mtfjsp_enc_head_tf32_grouped": ("h cand 2 6 36 sc sh 1 1 W bias 2 W1 b1 w2 b2 out S", "h W bias W1 sc sh", ""),
    "mtfjsp_enc_gat_trunk_tf32": ("f1 h W1 W2 W a_src a_dst out ws 72 S", "h W out", "f1 ws"),
    "mtfjsp_enc_gat_trunk_tf32_grouped": ("f1 h W1 W2 W a_src a_dst out ws 2 36 S", "h W out", "f1 ws"),
    "mtfjsp_enc_esa_mach_head_tf32": ("f1 h 2 36 W bias W1 b1 w2 b2 out S", "W bias W1", ""),
    "mtfjsp_enc_wgrad_tf32": ("g h 72 128 out b1 ws S", "g h ws", ""),
}
_BUFS = "h g out adj_w adj_src adj_dst sc sh w b mean rstd ws a_src a_dst parts W W1 W2 bias b1 w2 b2 cand f1".split()


def _abi_calls(base, stride):
    """(entry point, argument, alignment it needs, argument list with that buffer 4 bytes off) for every checked operand;
    buffer i sits at base + i * stride."""
    lib = _lib.lib()
    ptr = {n: base + i * stride for i, n in enumerate(_BUFS)}
    for fn, (args, a16, a8) in _ABI.items():
        for need, names in ((16, a16.split()), (8, a8.split())):
            for bad in names:
                vals = []
                for a, t in zip(args.split(), getattr(lib, fn).argtypes):
                    if a == "S":
                        vals.append(None)
                    elif a in ptr:
                        vals.append(C.c_void_p(ptr[a] + (4 if a == bad else 0)))
                    else:
                        vals.append(float(a) if t in (C.c_float, C.c_double) else int(a))
                yield fn, bad, need, vals


def test_misaligned_operands_are_refused_on_the_host():
    """Each 16-byte (and 8-byte) operand of each encoder entry point, 4 bytes off, returns MTFJSP_E_ARG.  The check
    runs on the host before any CUDA call, so the pointers are never dereferenced.  Without a GPU, the same calls with
    every pointer aligned get past the argument checks (they fail later, at the first CUDA call): so E_ARG above comes
    from the alignment check and not from another argument."""
    lib = _lib.lib()
    base, seen = 1 << 32, set()
    for fn, bad, need, vals in _abi_calls(base, 1 << 16):
        assert getattr(lib, fn)(*vals) == -1, (fn, bad)
        seen.add(fn)
    assert seen == set(_ABI)
    if not torch.cuda.is_available():
        for fn, (args, a16, a8) in _ABI.items():
            vals = next(v for f, _, _, v in _abi_calls(base, 1 << 16) if f == fn)
            vals = [C.c_void_p(v.value & ~15) if isinstance(v, C.c_void_p) else v for v in vals]
            assert getattr(lib, fn)(*vals) != -1, fn


@pytest.mark.gpu
def test_misaligned_device_operands_leave_every_buffer_untouched():
    """On the device: every buffer is a region of one NaN-filled allocation; each entry point called with one operand 4
    bytes off returns MTFJSP_E_ARG and writes nothing.  The test relies on the host-side alignment check and never
    launches a kernel: the calls return before any launch."""
    stride = 1 << 16  # floats per buffer, more than any of the calls could touch
    pool = torch.full((len(_BUFS) * stride + 64,), float("nan"), device="cuda")
    base = (pool.data_ptr() + 255) & ~255
    lib = _lib.lib()
    for fn, bad, need, vals in _abi_calls(base, stride * 4):
        assert getattr(lib, fn)(*vals) == -1, (fn, bad)
    torch.cuda.synchronize()
    assert bool(torch.isnan(pool).all())


def test_out_of_range_arguments_are_refused_on_the_host():
    """K outside 4 <= K <= 128, K % 4 == 0 (the grouped layer: K = 128 or 4 <= K <= 16), and an input scale without a
    shift, return MTFJSP_E_ARG before any CUDA call (dummy, aligned pointers)."""
    lib = _lib.lib()
    p = lambda i: C.c_void_p((1 << 32) + i * (1 << 16))
    for K in (0, 2, 6, 132):
        assert lib.mtfjsp_enc_linear_tf32(p(0), 64, K, p(1), p(2), None, None, 0, p(3), p(4), None) == -1, K
        assert lib.mtfjsp_enc_wgrad_tf32(p(0), p(1), 64, K, p(2), p(3), p(4), None) == -1, K
    for K in (0, 2, 6, 20, 64, 132):
        assert lib.mtfjsp_enc_linear_tf32_grouped(p(0), 2, 36, K, p(1), p(2), None, None, 0, 1, p(3), p(4), None) == -1, K
    # in_scale without in_shift
    assert lib.mtfjsp_enc_linear_tf32(p(0), 64, 128, p(1), p(2), p(5), None, 1, p(3), p(4), None) == -1
    assert lib.mtfjsp_enc_aggregate(p(0), p(1), p(2), p(3), 2, 36, 128, p(5), None, 1, None) == -1
    assert lib.mtfjsp_enc_graph_mean(p(0), p(3), 2, 36, 128, p(5), None, 1, None) == -1
    assert lib.mtfjsp_enc_aggregate_linear_tf32(p(0), 2, 36, p(1), p(2), p(6), p(7), p(5), None, 1, p(3), p(4), None) == -1
    assert lib.mtfjsp_enc_linear_tf32_grouped(p(0), 2, 36, 128, p(1), p(2), p(5), None, 1, 1, p(3), p(4), None) == -1
    assert lib.mtfjsp_enc_aggregate_linear_tf32_grouped(p(0), 2, 36, p(1), p(2), p(6), p(7), p(5), None, 1, 1, p(3), p(4),
                                                        None) == -1
    assert lib.mtfjsp_enc_head_tf32(p(0), p(1), 2, 6, 36, p(5), None, 1, p(6), p(7), 2, p(8), None, p(9), None, p(3), None) == -1
