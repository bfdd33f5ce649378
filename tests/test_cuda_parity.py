"""Parity tests proper: the sm_100a path, called through the C ABI, against
  (a) the committed reference dumps and the shipped result CSV rows (tests/golden),
  (b) the CPU oracle on the same seeded inputs at sizes it finishes in seconds,
  (c) size-independent schedule invariants at BASELINE.json's full batch sizes.
FP64 outputs are compared bit for bit; F32 observations must equal the oracle's FP64 value rounded once."""
import glob
import importlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle.mtfjsp_oracle import OracleEnv  # noqa: E402
from tests.test_oracle_golden import check_replay  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
eq = np.testing.assert_array_equal
SPEC_SIZES = ((6, 6), (10, 6), (20, 6), (10, 10), (15, 10), (20, 10), (30, 20))  # sizes with a specialised kernel


@pytest.fixture(params=["auto", "generic", "unfused", "fullobs"])
def kernel_path(request, monkeypatch):
    """'auto' = size-specialised kernel where one exists (random_step = one launch: policy + candidate-machine
    features + step + observation, observation rows rewritten incrementally after the first step of an episode);
    'unfused' = the same kernels with the pre-step kernel launched separately; 'fullobs' = every step rewrites the
    whole observation; 'generic' forces the one-warp-per-env kernel."""
    monkeypatch.setenv("MTFJSP_FORCE_GENERIC", "1" if request.param == "generic" else "0")
    monkeypatch.setenv("MTFJSP_FUSE_POLICY", "0" if request.param == "unfused" else "1")
    monkeypatch.setenv("MTFJSP_OBS_INCREMENTAL", "0" if request.param == "fullobs" else "1")
    return request.param


def _adapter():
    from tests import cuda_adapter

    return cuda_adapter


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("name", [os.path.basename(p) for p in sorted(glob.glob(os.path.join(GOLD, "replay_*.npz")))])
def test_replay_matches_reference_dump(name, fused, kernel_path):
    if kernel_path == "unfused":
        pytest.skip("recorded actions: no random_step here, 'auto' covers it")
    ad = _adapter()
    check_replay(lambda B, J, M, E, ls: ad.NumpyEnvAdapter(B, J, M, E, left_shift=ls, fused=fused), os.path.join(GOLD, name))


def test_pdr_rows_match_shipped_csv():
    ad = _adapter()
    g = np.load(os.path.join(GOLD, "pdr_golden.npz"))
    gold, ops, mch = g["gold"], g["ops"], g["mch"]
    R, S, N = ops.shape
    env = ad.NumpyEnvAdapter(S, 6, 6, 2, left_shift=False)
    env.load(g["t"], g["p"], g["transT"], g["edge"])
    env.scaler_init()
    w = np.tile(np.array([0.4, 0.4, 0.2]), (S, 1))
    for r in range(R):
        env.reset(w)
        for s in range(N):
            r5, s4, done, inv = env.step(ops[r, :, s], mch[r, :, s])
            assert not inv.any()
        assert done.all()
        eq(env.costs(), gold[r], err_msg=str(g["rule_names"][r]))


def _mk(B, J, M, E, seed, left_shift=True, dtype=torch.float64, mask_mode=1, scale=1.0, first_env=0):
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    d = ins.synthetic_instances(first_env, B, J, M, E, seed)
    t, tt = d["t"] * scale, d["transT"] * scale
    w = ins.random_weights(first_env, B, seed)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, obs_dtype=dtype, mask_mode=mask_mode)
    env.load(t, d["p"], tt, d["edge"])
    env.scaler_init()
    env.reset(w)
    ora = OracleEnv(B, J, M, E, left_shift=left_shift, nthreads=8)
    ora.load(t, d["p"], tt, d["edge"])
    ora.scaler_init()
    ora.reset(w)
    return env, ora, d, w


def _ell_to_dense(adj_w, adj_src):
    B, N, _ = adj_w.shape
    A = np.zeros((B, N, N))
    ar = np.arange(N)
    A[:, ar, ar] = 1.0
    bj, vj = np.nonzero(adj_w[:, :, 0])
    A[bj, vj, vj - 1] = adj_w[bj, vj, 0]
    bm, vm = np.nonzero(adj_src >= 0)
    A[bm, vm, adj_src[bm, vm]] = adj_w[bm, vm, 1]
    return A


@pytest.mark.parametrize("cfg", [
    # B, J, M, E, left_shift, mask_mode, scale, episodes
    (512, 6, 6, 2, True, 1, 1.0, 2),
    (512, 6, 6, 2, True, 0, 1.0, 1),
    (256, 6, 6, 2, False, 0, 1.0, 1),
    (256, 6, 6, 2, True, 0, 0.02, 1),
    (128, 10, 10, 3, True, 1, 1.0, 1),
    (128, 10, 10, 3, True, 0, 1.0, 1),
    (64, 3, 4, 2, True, 0, 1.0, 2),
    (33, 2, 2, 1, True, 0, 1.0, 1),
    (40, 20, 5, 2, True, 0, 1.0, 1),
    (24, 5, 33, 4, True, 0, 1.0, 1),
    (16, 30, 20, 5, True, 0, 1.0, 1),
    (16, 30, 20, 5, True, 1, 1.0, 1),
    (7, 30, 20, 5, False, 0, 1.0, 1),
    (65, 10, 10, 3, False, 0, 1.0, 1),
    (1, 6, 6, 2, True, 1, 1.0, 1),
    (3, 6, 6, 2, True, 0, 1.0, 1),
    (8, 40, 8, 2, True, 0, 0.05, 1),
    # the other sizes of the reference's instance generator (generate_allsize_mofjsp_dataset.py:429), specialised kernels
    (33, 10, 6, 2, True, 1, 1.0, 2),
    (17, 20, 6, 3, True, 1, 1.0, 1),
    (13, 15, 10, 2, True, 1, 1.0, 1),
    (13, 15, 10, 2, False, 0, 1.0, 1),
    (9, 20, 10, 5, True, 1, 1.0, 1),
])
def test_random_rollout_matches_oracle_every_step(cfg, kernel_path):
    B, J, M, E, ls, mm, scale, episodes = cfg
    if kernel_path != "auto" and (J, M) not in SPEC_SIZES:
        pytest.skip("size has no specialised kernel: 'auto' already ran the generic one")
    N = J * M
    env, ora, d, w = _mk(B, J, M, E, seed=1000 + J * M, left_shift=ls, mask_mode=mm, scale=scale)
    ob = ora.obs(mm)
    env.obs(mm)
    eq(env.task_fea.cpu().numpy(), ob["task_fea"])
    eq(env.job_mask.cpu().numpy(), ob["job_mask"])
    for ep in range(episodes):
        if ep > 0:
            w2 = ins.random_weights(0, B, 77 + ep)
            env.reset(w2); ora.reset(w2)
            env.scaler_reset(); ora.scaler_reset()
        for s in range(N):
            env.random_step(seed=42 + ep, env_offset=0, mask_mode=mm)
            op, mc = env.op.cpu().numpy(), env.mach.cpu().numpy()
            # the device policy draws the same counter-based action as the oracle's policy
            m1, mmask = ora.mfea1(op)
            r5, s4, done, inv = ora.step(op, mc)
            assert not inv.any(), (s, op[inv.astype(bool)], mc[inv.astype(bool)])
            ob = ora.obs(mm)
            eq(env.invalid.cpu().numpy(), inv)
            eq(env.mfea1_buf.cpu().numpy(), m1)
            eq(env.mach_mask.cpu().numpy(), mmask)
            eq(env.reward5.cpu().numpy(), r5)
            eq(env.scaled4.cpu().numpy(), s4)
            eq(env.done.cpu().numpy(), done)
            eq(env.task_fea.cpu().numpy(), ob["task_fea"])
            eq(env.mach_fea.cpu().numpy(), ob["mach_fea"])
            eq(env.job_mask.cpu().numpy(), ob["job_mask"])
            eq(env.candidate.cpu().numpy(), ob["candidate"])
            if s % 7 == 0 or s == N - 1:
                eq(_ell_to_dense(env.adj_w.cpu().numpy().astype(np.float64), env.adj_src.cpu().numpy().astype(np.int64)),
                   ora.dense_adj())
                st = {k: v.cpu().numpy() for k, v in env.export_state().items()}
                so = ora.export_state()
                for k in so:
                    eq(st[k], so[k], err_msg=k)
        assert env.done.cpu().numpy().all()
        eq(env.costs().cpu().numpy(), ora.costs())
        sc, so = env.export_scaler(), ora.export_scaler()
        for k in so:
            eq(sc[k].cpu().numpy(), so[k], err_msg=k)


def test_oracle_policy_replays_device_actions():
    """oracle_rollout_random (the CPU baseline loop) draws exactly the actions the device policy draws."""
    B, J, M, E = 256, 6, 6, 2
    env, ora, d, w = _mk(B, J, M, E, seed=5)
    acts = []
    for s in range(J * M):
        env.random_step(seed=9, env_offset=0)
        acts.append(np.stack([env.op.cpu().numpy(), env.mach.cpu().numpy()], 1))
    out = ora.rollout_random(J * M, seed=9, env_offset=0, mask_mode=1, record_actions=True)
    eq(out["actions"], np.stack(acts))
    eq(env.task_fea.cpu().numpy(), out["task_fea"])
    eq(env.reward5.cpu().numpy(), out["reward5"])


def test_f32_observations_are_the_rounded_f64_values():
    B, J, M, E = 256, 6, 6, 2
    env, ora, d, w = _mk(B, J, M, E, seed=11, dtype=torch.float32)
    for s in range(J * M):
        env.random_step(seed=3)
        op, mc = env.op.cpu().numpy(), env.mach.cpu().numpy()
        m1, _ = ora.mfea1(op)
        ora.step(op, mc)
        ob = ora.obs(1)
        eq(env.task_fea.cpu().numpy(), ob["task_fea"].astype(np.float32))
        eq(env.mach_fea.cpu().numpy(), ob["mach_fea"].astype(np.float32))
        eq(env.mfea1_buf.cpu().numpy(), m1.astype(np.float32))
    eq(env.dense_adj(torch.float32).cpu().numpy(), ora.dense_adj().astype(np.float32))


def test_invalid_actions_are_flagged_and_leave_state_untouched():
    B, J, M, E = 64, 3, 3, 1
    env, ora, d, w = _mk(B, J, M, E, seed=5)
    dev = env.device
    i32 = lambda x: torch.as_tensor(np.asarray(x, dtype=np.int32)).to(dev)
    before = {k: v.cpu().numpy() for k, v in env.export_state().items()}
    feas = np.argmax(d["t"][:, 0] >= 0, axis=1)
    for op, mc in ((np.full(B, 1), feas), (np.full(B, 99), feas), (np.zeros(B), np.full(B, 7)), (np.full(B, -1), feas)):
        env.step(i32(op), i32(mc))
        assert env.invalid.cpu().numpy().all()
        eq(env.reward5.cpu().numpy(), 0.0)
    after = {k: v.cpu().numpy() for k, v in env.export_state().items()}
    for k in before:
        eq(before[k], after[k])
    env.step(i32(np.zeros(B)), i32(feas))
    assert not env.invalid.cpu().numpy().any()
    env.step(i32(np.zeros(B)), i32(feas))
    assert env.invalid.cpu().numpy().all()
    infeas = np.argmax(d["t"][:, 1] < 0, axis=1)
    env.step(i32(np.ones(B)), i32(infeas))
    eq(env.invalid.cpu().numpy().astype(bool), (d["t"][:, 1] < 0).any(axis=1))


def test_step_before_reset_is_a_state_error():
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    lib = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")
    env = envm.BatchedMTFJSPEnv(4, 3, 3, 1)
    with pytest.raises(lib.MTFJSPError):
        env.step(env.op, env.mach)


@pytest.mark.parametrize("B", [4096 + 77, 3 * 4096 + 77])
@pytest.mark.parametrize("pinned", [True, False, "mixed", "zerocopy_actions"])
def test_host_step_equals_device_step(pinned, B, kernel_path, monkeypatch):
    """mtfjsp_step_host and mtfjsp_step_host_packed with pinned host buffers (one launch that writes step info, job mask,
    candidates and records straight into the mapped host buffers; with the generic kernel under kernel_path "generic")
    and with pageable ones (copy in, launch, copy out) must equal the device-pointer call bit for bit, including the
    all-invalid step after the episode has ended.  "mixed" = pageable actions with pinned outputs: one pageable buffer
    sends the whole call the staged way.  "zerocopy_actions" = the actions are read from the mapped host buffers in
    place as well (MTFJSP_HOST_ZEROCOPY=2; by default only from 16,384 envs up)."""
    if kernel_path == "unfused":
        pytest.skip("no random_step here, 'auto' covers it")
    if pinned == "zerocopy_actions":
        monkeypatch.setenv("MTFJSP_HOST_ZEROCOPY", "2")  # read by mtfjsp_create
        pinned = True
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    J, M, E = 6, 6, 2
    N = J * M
    d = ins.synthetic_instances(0, B, J, M, E, 77)
    w = ins.random_weights(0, B, 77)
    envs = []
    for _ in range(2):
        env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
        env.load(d["t"], d["p"], d["transT"], d["edge"])
        env.scaler_init()
        env.reset(w)
        envs.append(env)
    dev_env, host_env = envs
    pk_env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)  # packed-record form
    pk_env.load(d["t"], d["p"], d["transT"], d["edge"])
    pk_env.scaler_init()
    pk_env.reset(w)
    io_env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)  # step info only comes back
    io_env.load(d["t"], d["p"], d["transT"], d["edge"])
    io_env.scaler_init()
    io_env.reset(w)
    pk_act, pk_rec = pk_env.host_buffers()
    if pinned is not True:
        pk_act = pk_act.clone()
    if not pinned:
        pk_rec = pk_rec.clone()
    assert pk_act.is_pinned() == (pinned is True) and pk_rec.is_pinned() == bool(pinned)
    pk_rec.fill_(0xAB)
    pin_in = (lambda x: x.pin_memory()) if pinned is True else (lambda x: x)
    pin = (lambda x: x.pin_memory()) if pinned else (lambda x: x)
    info6 = pin(torch.full((B, 6), -7.0, dtype=torch.float64))
    h_jm = pin(torch.full((B, J), 9, dtype=torch.uint8))
    h_cd = pin(torch.full((B, J), -1, dtype=torch.int32))
    info6_only = pin(torch.full((B, 6), -9.0, dtype=torch.float64))
    for s in range(N + 1):  # one step past the end: every action is invalid and must be reported as such
        op, mach = dev_env.policy_random(seed=5)
        if s == N:
            op, mach = torch.zeros_like(op), torch.zeros_like(mach)
        h_op, h_mc = pin_in(op.cpu()), pin_in(mach.cpu())
        dev_env.step_obs(op, mach)
        host_env.step_host(h_op, h_mc, info6, h_jm, h_cd)
        eq(info6[:, 0].numpy(), dev_env.reward5[:, 0].cpu().numpy())
        eq(info6[:, 1].numpy(), dev_env.done.cpu().numpy().astype(np.float64))
        eq(info6[:, 2:].numpy(), dev_env.scaled4.cpu().numpy())
        eq(h_jm.numpy(), dev_env.job_mask.cpu().numpy())
        eq(h_cd.numpy(), dev_env.candidate.cpu().numpy())
        io_env.step_host(h_op, h_mc, info6_only, None, None)
        eq(info6_only.numpy(), info6.numpy())
        pk_act[:, 0].copy_(op.cpu()); pk_act[:, 1].copy_(mach.cpu())
        if s % 2:   # the prepared-call form and the general method are interchangeable
            pk_env.host_stepper(pk_rec)(pk_act.data_ptr())
        else:
            pk_env.step_host_packed(pk_act, pk_rec)
        r_info6, r_cand, r_mask = pk_env.decode_records(pk_rec)
        eq(r_info6, info6.numpy())
        eq(r_cand, h_cd.numpy())
        eq(r_mask, h_jm.numpy())
        raw = pk_rec.numpy()
        used = 41 + (J + 7) // 8 + J
        assert not raw[:, used:].any()   # padding is written (zero), never left over
        for name in ("task_fea", "mach_fea", "adj_w", "adj_src"):
            assert torch.equal(getattr(host_env, name), getattr(dev_env, name)), (name, s)
            assert torch.equal(getattr(pk_env, name), getattr(dev_env, name)), (name, s)
            assert torch.equal(getattr(io_env, name), getattr(dev_env, name)), (name, s)
        assert int(dev_env.invalid.sum()) == (B if s == N else 0)
    assert bool(dev_env.done.all()) and float(info6[:, 1].sum()) == B
    eq(host_env.costs().cpu().numpy(), dev_env.costs().cpu().numpy())
    eq(pk_env.costs().cpu().numpy(), dev_env.costs().cpu().numpy())


@pytest.mark.parametrize("B", [1, 2, 3, 5, 17])
def test_packed_host_records_tiny_batches(B):
    """Batches smaller than a warp's four envs (and not a multiple of it): the whole-warp record runs stop at the batch's
    end, nothing is written behind it."""
    J, M, E = 6, 6, 2
    N = J * M
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    d = ins.synthetic_instances(0, B, J, M, E, 13)
    w = ins.random_weights(0, B, 13)
    envs = []
    for _ in range(2):
        env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
        env.load(d["t"], d["p"], d["transT"], d["edge"])
        env.scaler_init()
        env.reset(w)
        envs.append(env)
    dev_env, pk_env = envs
    nbytes = int(pk_env.host_buffers()[1].shape[1])
    pk_act = torch.zeros((B, 2), dtype=torch.int32).pin_memory()
    guard = torch.full((B + 4, nbytes), 0x5A, dtype=torch.uint8).pin_memory()   # four records of canary behind the batch
    pk_rec = guard[:B]
    info6_only = torch.full((B + 2, 6), -9.0, dtype=torch.float64).pin_memory()
    for s in range(N):
        op, mach = dev_env.policy_random(seed=4)
        dev_env.step_obs(op, mach)
        pk_act[:, 0].copy_(op.cpu()); pk_act[:, 1].copy_(mach.cpu())
        pk_env.step_host_packed(pk_act, pk_rec)
        info6, cand, mask = pk_env.decode_records(pk_rec)
        eq(info6[:, 0], dev_env.reward5[:, 0].cpu().numpy())
        eq(info6[:, 2:], dev_env.scaled4.cpu().numpy())
        eq(cand, dev_env.candidate.cpu().numpy())
        eq(mask, dev_env.job_mask.cpu().numpy())
        assert bool((guard[B:] == 0x5A).all())
    assert bool(dev_env.done.all())
    io_env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    io_env.load(d["t"], d["p"], d["transT"], d["edge"])
    io_env.scaler_init()
    io_env.reset(w)
    dev_env.reset(w); dev_env.scaler_reset(); io_env.scaler_reset()
    op, mach = dev_env.policy_random(seed=6)
    dev_env.step_obs(op, mach)
    io_env.step_host(op.cpu().pin_memory(), mach.cpu().pin_memory(), info6_only[:B], None, None)
    eq(info6_only[:B, 0].numpy(), dev_env.reward5[:, 0].cpu().numpy())
    assert bool((info6_only[B:] == -9.0).all())


@pytest.mark.parametrize("size", [(10, 10, 3), (20, 6, 3), (15, 10, 2), (30, 20, 5), (3, 4, 2), (9, 5, 1)])
def test_packed_host_records_other_sizes(size):
    """Packed host-step records at sizes with odd record word counts, more than 8 jobs (several mask bytes), the COLD /
    NOTT kernels, and sizes without a specialised kernel: decoded records equal the device-pointer call's outputs."""
    J, M, E = size
    N, B = J * M, 333
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    d = ins.synthetic_instances(0, B, J, M, E, 91)
    w = ins.random_weights(0, B, 91)
    envs = []
    for _ in range(2):
        env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
        env.load(d["t"], d["p"], d["transT"], d["edge"])
        env.scaler_init()
        env.reset(w)
        envs.append(env)
    dev_env, pk_env = envs
    pk_act, pk_rec = pk_env.host_buffers()
    assert pk_rec.shape[1] == (41 + (J + 7) // 8 + J + 7) // 8 * 8
    pk_rec.fill_(0xCD)
    steps = list(range(N)) if N <= 150 else list(range(40)) + list(range(N - 3, N))
    for s in range(N):
        op, mach = dev_env.policy_random(seed=17)
        dev_env.step_obs(op, mach)
        pk_act[:, 0].copy_(op.cpu()); pk_act[:, 1].copy_(mach.cpu())
        pk_env.step_host_packed(pk_act, pk_rec)
        if s not in steps:
            continue
        info6, cand, mask = pk_env.decode_records(pk_rec)
        eq(info6[:, 0], dev_env.reward5[:, 0].cpu().numpy())
        eq(info6[:, 1], dev_env.done.cpu().numpy().astype(np.float64))
        eq(info6[:, 2:], dev_env.scaled4.cpu().numpy())
        eq(cand, dev_env.candidate.cpu().numpy())
        eq(mask, dev_env.job_mask.cpu().numpy())
        assert not pk_rec.numpy()[:, 41 + (J + 7) // 8 + J:].any()
        for name in ("task_fea", "mach_fea", "adj_w", "adj_src"):
            assert torch.equal(getattr(pk_env, name), getattr(dev_env, name)), (name, s)
    assert bool(dev_env.done.all())


@pytest.mark.parametrize("cfg", [(65536, 6, 6, 2), (16384, 10, 10, 3), (4096, 30, 20, 5)])
def test_full_size_rollout_invariants(cfg):
    """BASELINE.json sizes: schedule invariants + telescoping rewards + a replay-checked random subset."""
    B, J, M, E = cfg
    N = J * M
    envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
    d = ins.synthetic_instances(0, B, J, M, E, 1000 + N)
    w = ins.random_weights(0, B, 1000 + N)
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    c0 = env.costs().clone()
    rsum = torch.zeros((B, 5), dtype=torch.float64, device=env.device)
    rng = np.random.default_rng(0)
    sub = np.sort(rng.choice(B, 1024 if N <= 100 else 128, replace=False))
    acts = np.zeros((N, len(sub), 2), dtype=np.int32)
    for s in range(N):
        env.random_step(seed=123, env_offset=0)
        rsum += env.reward5
        acts[s, :, 0] = env.op.cpu().numpy()[sub]
        acts[s, :, 1] = env.mach.cpu().numpy()[sub]
        assert int(env.invalid.sum().item()) == 0
        assert int(env.done.sum().item()) == (B if s == N - 1 else 0)
    c1 = env.costs()
    # rewards telescope to (initial estimate - final cost) per component (SS:1066-1088)
    tot = rsum.cpu().numpy()
    np.testing.assert_allclose(tot[:, 1], (c0[:, 0] - c1[:, 0]).cpu().numpy(), rtol=1e-9, atol=1e-7)
    np.testing.assert_allclose(tot[:, 3], (c0[:, 1] - c1[:, 1]).cpu().numpy(), rtol=1e-9, atol=1e-7)
    np.testing.assert_allclose(tot[:, 4], -c1[:, 2].cpu().numpy(), rtol=1e-9, atol=1e-7)
    np.testing.assert_allclose(tot[:, 2], -c1[:, 3].cpu().numpy(), rtol=1e-9, atol=1e-6)
    st = {k: v.cpu().numpy() for k, v in env.export_state().items()}
    mach, stt, ftt, routes = st["mach"], st["st"], st["ft"], st["routes"]
    assert (mach >= 0).all()
    t = d["t"]
    dur = np.take_along_axis(t, mach[:, :, None].astype(np.int64), axis=2)[:, :, 0]
    assert (dur > 0).all()
    eq(ftt, stt + dur)                                    # ft = st + dur, machine feasible
    s2, f2 = stt.reshape(B, J, M), ftt.reshape(B, J, M)
    assert (s2[:, :, 1:] >= f2[:, :, :-1]).all()          # job precedence
    assert ((routes >= 0).sum(axis=(1, 2)) == N).all()    # every op on exactly one route
    for m in range(M):                                    # no overlap on a machine, route order = time order
        r = routes[:, m, :]
        ok = r >= 0
        rs = np.where(ok, np.take_along_axis(stt, np.maximum(r, 0).astype(np.int64), 1), np.inf)
        rf = np.where(ok, np.take_along_axis(ftt, np.maximum(r, 0).astype(np.int64), 1), np.inf)
        nxt_ok = ok[:, 1:]
        assert (rs[:, 1:][nxt_ok] >= rf[:, :-1][nxt_ok]).all()
        mm_ = np.where(ok, np.take_along_axis(mach, np.maximum(r, 0).astype(np.int64), 1), m)
        assert (mm_ == m).all()
    eq(c1[:, 0].cpu().numpy(), ftt.max(axis=1))           # final makespan is the true one
    # replay the recorded actions of a random subset on the oracle: bit-exact schedules and costs
    ora = OracleEnv(len(sub), J, M, E, left_shift=True, nthreads=8)
    ora.load(t[sub], d["p"][sub], d["transT"][sub], d["edge"][sub])
    ora.scaler_init()
    ora.reset(w[sub])
    for s in range(N):
        r5, s4, done, inv = ora.step(acts[s, :, 0], acts[s, :, 1])
        assert not inv.any()
    so = ora.export_state()
    eq(mach[sub], so["mach"]); eq(stt[sub], so["st"]); eq(ftt[sub], so["ft"]); eq(routes[sub], so["routes"])
    eq(c1.cpu().numpy()[sub], ora.costs())
    eq(env.reward5.cpu().numpy()[sub], r5)
    eq(env.scaled4.cpu().numpy()[sub], s4)
    ob = ora.obs(1)
    eq(env.task_fea.cpu().numpy()[sub], ob["task_fea"].astype(np.float32))


def test_incremental_observation_bookkeeping():
    """The incremental observation may only be used while the SAME output buffers have followed every step since a full
    observation.  Break the chain in every way the C ABI allows -- other buffers, a step without observation, a reset, a
    side view (dense_adj), an invalid action -- and compare the buffers with the oracle after every step."""
    B, J, M, E = 200, 6, 6, 2
    N = J * M
    env, ora, d, w = _mk(B, J, M, E, seed=11, dtype=torch.float32)
    main = (env.task_fea, env.mach_fea, env.adj_w, env.adj_src)
    other = tuple(torch.full_like(x, 77) for x in main)

    def check(tag):
        ob = ora.obs(1)
        eq(env.task_fea.cpu().numpy(), ob["task_fea"].astype(np.float32), err_msg=tag)
        eq(env.mach_fea.cpu().numpy(), ob["mach_fea"].astype(np.float32), err_msg=tag)
        eq(_ell_to_dense(env.adj_w.cpu().numpy().astype(np.float64), env.adj_src.cpu().numpy().astype(np.int64)),
           ora.dense_adj(), err_msg=tag)

    def use(bufs):
        env.task_fea, env.mach_fea, env.adj_w, env.adj_src = bufs

    for s in range(N):
        op, mach = env.policy_random(seed=3)
        o, m = op.cpu().numpy().copy(), mach.cpu().numpy().copy()
        if s == 5:      # other buffers (filled with garbage): must be rewritten completely
            use(other)
        if s == 9:      # ... and back to the main ones, which are 4 steps stale by now
            use(main)
        if s == 12:     # a step without observation breaks the chain
            env.step(op, mach); ora.step(o, m)
            op, mach = env.policy_random(seed=4)
            o, m = op.cpu().numpy().copy(), mach.cpu().numpy().copy()
        if s == 15:     # a side view into other memory must not disturb the chain
            env.dense_adj()
        if s == 20:     # invalid actions for half of the envs: their state and rows stay as they are
            op = op.clone(); op[::2] = -1
            o = op.cpu().numpy().copy()
        env.step_obs(op, mach)
        r5, s4, done, inv = ora.step(o, m)
        eq(env.invalid.cpu().numpy(), inv)
        check("step %d" % s)
    w2 = ins.random_weights(0, B, 99)
    env.reset(w2); ora.reset(w2)          # a reset breaks the chain: the first step of the episode writes everything
    env.random_step(seed=8)
    ora.step(env.op.cpu().numpy(), env.mach.cpu().numpy())
    check("after reset")
