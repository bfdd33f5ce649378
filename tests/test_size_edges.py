"""The environment at the edges of its size range (include/mtfjsp.h: 2 <= M <= 64, J >= 1, and one env's state within
one block's shared memory), where one-warp-per-env kernels go wrong: more machines than lanes (64-bit machine masks),
one job (the ESA mask's one-job branches), more jobs than lanes (32-job chunks, several mask bytes, ~2 KB host
records), one transport group per machine, and N in the thousands (32 pairwise-sum leaves, ~100 idle-sum prefixes, one
warp per block using ~225 KB of shared memory).

Instances come from `reference_stream_instances`: the other two generators cannot make these sizes (the Philox one
draws whole 1024-env blocks, the device one needs J >= M).  FP64 outputs are compared with the CPU oracle bit for bit;
F32 observations must equal the oracle's FP64 values rounded once."""
import ctypes as C
import importlib
import os
import re
import time

import numpy as np
import pytest

from oracle.mtfjsp_oracle import OracleEnv, rand_u32

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
eq = np.testing.assert_array_equal
FIN, ESA = 0, 1
E_ARG = -1

# largest J that mtfjsp_create accepts at each M (B = 1); the header states the same numbers
CREATE_MAX_J = {2: 1678, 3: 1152, 7: 510, 32: 109, 33: 106, 64: 48}


def test_header_states_the_create_limits():
    """include/mtfjsp.h names the largest J per M that the boundary test below finds on the device."""
    with open(os.path.join(ROOT, "include", "mtfjsp.h")) as f:
        text = f.read()
    stated = {int(m): int(j) for m, j in re.findall(r"M = (\d+): J <= (\d+)", text)}
    assert stated == CREATE_MAX_J


def _torch():
    return pytest.importorskip("torch")


def _envm():
    return importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")


def _libm():
    return importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")


def _create_rc(B, J, M, E=1):
    """Return code of mtfjsp_create for this size; a handle it made is destroyed at once."""
    torch = _torch()
    lib = _libm().lib()
    h = C.c_void_p()
    rc = lib.mtfjsp_create(C.byref(h), B, J, M, E, 1, torch.cuda.current_device())
    if rc == 0:
        assert h.value
        lib.mtfjsp_destroy(h)
    else:
        assert not h.value
    return rc


# ---------------------------------------------------------------------------------------------------------------------
# oracle parity, one random episode after another
# ---------------------------------------------------------------------------------------------------------------------

def _ell_matches_dense(adj_w, adj_src, dense, M, tag):
    """The compact ELL rows (job-predecessor weight, machine-predecessor source and weight, implicit diagonal 1) hold
    exactly the nonzero entries of the dense [B, dst, src] matrix -- checked without building a second N x N array."""
    B, N, _ = adj_w.shape
    ar = np.arange(N)
    eq(dense[:, ar, ar], 1.0, err_msg=tag)
    wj = adj_w[:, :, 0].astype(np.float64)
    eq(wj[:, ar % M == 0], 0.0, err_msg=tag)                # a job's first op has no job predecessor
    prev_is_src = adj_src == ar[None, :] - 1                 # machine predecessor v - 1 of another job (or no job arc)
    eq(wj[prev_is_src], 0.0, err_msg=tag)
    bj, vj = np.nonzero((ar % M != 0)[None, :] & ~prev_is_src)
    eq(dense[bj, vj, vj - 1], wj[bj, vj], err_msg=tag)
    bm, vm = np.nonzero(adj_src >= 0)
    eq(dense[bm, vm, adj_src[bm, vm]], adj_w[bm, vm, 1].astype(np.float64), err_msg=tag)
    eq(np.count_nonzero(dense, axis=2), 1 + (wj != 0) + (adj_src >= 0), err_msg=tag)


def _expected_random_action(ora_mask, cand, t, seed, env_offset, step):
    """The counter-based random policy (include/mtfjsp.h, mtfjsp_policy_random) restated per env: the k-th selectable
    job's candidate op, then the km-th feasible machine of that op."""
    B = ora_mask.shape[0]
    op = np.full(B, -1, dtype=np.int32)
    mc = np.full(B, -1, dtype=np.int32)
    for b in range(B):
        free = np.flatnonzero(ora_mask[b] == 0)
        if len(free) == 0:
            continue
        k = (rand_u32(seed, env_offset + b, step, 0) * len(free)) >> 32
        op[b] = cand[b, free[k]]
        feas = np.flatnonzero(t[b, op[b]] >= 0)
        km = (rand_u32(seed, env_offset + b, step, 1) * len(feas)) >> 32
        mc[b] = feas[km]
    return op, mc


def _checkpoints(N):
    """About 16 spread steps plus the last five."""
    return sorted(set(np.linspace(0, N - 1, 16).astype(int).tolist()) | set(range(max(0, N - 5), N)))


def _run_parity(B, J, M, E, left_shift, mask_mode, f32, seed, episodes=2, env_offset=0):
    torch = _torch()
    N = J * M
    dtype = torch.float32 if f32 else torch.float64
    cast = (lambda x: x.astype(np.float32)) if f32 else (lambda x: x)
    d = ins.reference_stream_instances(B, J, M, E, seed)
    t = d["t"]
    w = ins.random_weights(0, B, seed)
    env = _envm().BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, obs_dtype=dtype, mask_mode=mask_mode)
    env.load(t, d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    ora = OracleEnv(B, J, M, E, left_shift=left_shift, nthreads=8)
    ora.load(t, d["p"], d["transT"], d["edge"])
    ora.scaler_init()
    ora.reset(w)
    ob = ora.obs(mask_mode)
    env.obs(mask_mode)
    eq(env.task_fea.cpu().numpy(), cast(ob["task_fea"]))
    eq(env.mach_fea.cpu().numpy(), cast(ob["mach_fea"]))
    eq(env.job_mask.cpu().numpy(), ob["job_mask"])
    eq(env.candidate.cpu().numpy(), ob["candidate"])
    check_at = set(_checkpoints(N))
    for ep in range(episodes):
        if ep > 0:
            w2 = ins.random_weights(0, B, seed, episode=ep)
            env.reset(w2); ora.reset(w2)
            env.scaler_reset(); ora.scaler_reset()
            ob = ora.obs(mask_mode)
        pseed = 42 + ep
        for s in range(N):
            want_op, want_mc = _expected_random_action(ob["job_mask"], ob["candidate"], t, pseed, env_offset, s)
            env.random_step(seed=pseed, env_offset=env_offset, mask_mode=mask_mode)
            op, mc = env.op.cpu().numpy(), env.mach.cpu().numpy()
            tag = "episode %d step %d" % (ep, s)
            eq(op, want_op, err_msg=tag)
            eq(mc, want_mc, err_msg=tag)
            m1, mmask = ora.mfea1(op)
            r5, s4, done, inv = ora.step(op, mc)
            assert not inv.any(), tag
            ob = ora.obs(mask_mode)
            eq(env.invalid.cpu().numpy(), inv, err_msg=tag)
            eq(env.mfea1_buf.cpu().numpy(), cast(m1), err_msg=tag)
            eq(env.mach_mask.cpu().numpy(), mmask, err_msg=tag)
            eq(env.reward5.cpu().numpy(), r5, err_msg=tag)
            eq(env.scaled4.cpu().numpy(), s4, err_msg=tag)
            eq(env.done.cpu().numpy(), done, err_msg=tag)
            eq(env.task_fea.cpu().numpy(), cast(ob["task_fea"]), err_msg=tag)
            eq(env.mach_fea.cpu().numpy(), cast(ob["mach_fea"]), err_msg=tag)
            eq(env.job_mask.cpu().numpy(), ob["job_mask"], err_msg=tag)
            eq(env.candidate.cpu().numpy(), ob["candidate"], err_msg=tag)
            if s in check_at:
                _ell_matches_dense(env.adj_w.cpu().numpy(), env.adj_src.cpu().numpy().astype(np.int64), ora.dense_adj(),
                                   M, tag)
                st = {k: v.cpu().numpy() for k, v in env.export_state().items()}
                so = ora.export_state()
                for k in so:
                    eq(st[k], so[k], err_msg="%s %s" % (tag, k))
        assert env.done.cpu().numpy().all()
        eq(env.costs().cpu().numpy(), ora.costs())
        sc, so = env.export_scaler(), ora.export_scaler()
        for k in so:
            eq(sc[k].cpu().numpy(), so[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.parametrize("M", sorted(CREATE_MAX_J))
def test_create_accepts_exactly_up_to_the_stated_size(M):
    """Bisection on mtfjsp_create: every J up to the table's value is accepted, the next one is refused with
    MTFJSP_E_ARG (the per-env state no longer fits one block's shared memory), and the library stays usable."""
    lo, hi = 1, 4096 // M + 1          # create accepts lo, refuses hi (N > 4096 always is)
    assert _create_rc(1, lo, M) == 0 and _create_rc(1, hi, M) == E_ARG
    while hi - lo > 1:
        mid = (lo + hi) // 2
        rc = _create_rc(1, mid, M)
        assert rc in (0, E_ARG), rc
        if rc == 0:
            lo = mid
        else:
            hi = mid
    assert lo == CREATE_MAX_J[M]
    for B in (1, 64):                   # the limit is per env: it does not move with the batch size
        assert _create_rc(B, lo, M, E=M) == 0
        assert _create_rc(B, lo + 1, M, E=M) == E_ARG
    lib = _libm()
    with pytest.raises(lib.MTFJSPError, match=r"\(-1\).*shared memory"):
        _envm().BatchedMTFJSPEnv(1, lo + 1, M, 1)
    _run_parity(4, 6, 6, 2, True, ESA, False, seed=5, episodes=1)


@pytest.mark.gpu
def test_create_rejects_sizes_outside_the_range():
    for B, J, M, E in ((1, 4, 1, 1), (1, 4, 65, 1), (1, 1, 65, 65), (1, 0, 6, 2), (0, 6, 6, 2), (1, 6, 6, 0),
                       (1, 65, 64, 4), (1, 2049, 2, 1), (1, 4096, 1, 1),
                       (1, 64, 64, 4), (1, 2048, 2, 1), (1, 128, 32, 4)):   # N = 4096 never fits shared memory
        assert _create_rc(B, J, M, E) == E_ARG, (B, J, M, E)
    assert _create_rc(1, 1, 64, 64) == 0 and _create_rc(1, 1, 2, 1) == 0
    _run_parity(3, 3, 4, 2, False, FIN, True, seed=6, episodes=1)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [
    # B, J, M, E, left_shift, mask_mode, f32, incremental observation
    (3, 48, 64, 4, True, ESA, False, True),
    (3, 48, 64, 64, False, FIN, True, False),
    (3, 106, 33, 5, True, FIN, True, True),
    (3, 106, 33, 2, False, ESA, False, False),
    (3, 1678, 2, 1, True, ESA, True, False),
    (3, 1678, 2, 2, False, FIN, False, True),
    (3, 1, 64, 7, True, ESA, False, False),
    (5, 1, 64, 64, False, FIN, True, True),
    (5, 1, 64, 1, True, ESA, True, False),
    (3, 1, 2, 1, False, ESA, True, True),
    (5, 1, 2, 2, True, FIN, False, False),
    (5, 1, 2, 1, False, ESA, False, True),
], ids=lambda c: "B%dJ%dM%dE%d_%s_%s_%s_%s" % (c[0], c[1], c[2], c[3], "ls" if c[4] else "nols", "esa" if c[5] else "fin",
                                              "f32" if c[6] else "f64", "inc" if c[7] else "full"))
def test_largest_sizes_match_the_oracle_every_step(cfg, monkeypatch):
    """The largest J create accepts at M = 64, 33 and 2, and J = 1 at M = 64 and 2: two random episodes (the second
    after reset + scaler_reset) against the oracle after every step; adjacency and schedule state at spread steps."""
    B, J, M, E, ls, mm, f32, inc = cfg
    monkeypatch.setenv("MTFJSP_OBS_INCREMENTAL", "1" if inc else "0")   # read by mtfjsp_create
    monkeypatch.setenv("MTFJSP_FORCE_GENERIC", "0")
    t0 = time.perf_counter()
    _run_parity(B, J, M, E, ls, mm, f32, seed=2000 + J * M + E, env_offset=B * 7)
    print("%s: %.1f s" % (cfg, time.perf_counter() - t0))


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(48, 64, 4), (1678, 2, 1), (106, 33, 3)])
def test_views_at_large_n(size):
    """dense_adj (F64 and F32) and raw_adj of one env mid-episode.  The dense view is the observation's adjacency,
    adj[v, u] with diagonal 1; raw_adj holds the graph's arc weights truncated towards zero, adj[u, v] (source-major),
    no diagonal.  They describe the same arcs: an arc's weight is its source's duration plus transport and waiting time
    (at least that duration) once the source is scheduled, and 1 from an unscheduled job predecessor."""
    torch = _torch()
    J, M, E = size
    N = J * M
    d = ins.reference_stream_instances(1, J, M, E, 31)
    w = ins.random_weights(0, 1, 31)
    env = _envm().BatchedMTFJSPEnv(1, J, M, E, left_shift=True, obs_dtype=torch.float64)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    ora = OracleEnv(1, J, M, E, left_shift=True, nthreads=8)
    ora.load(d["t"], d["p"], d["transT"], d["edge"])
    ora.scaler_init()
    ora.reset(w)
    for s in range(N // 2 + 1):
        env.random_step(seed=8)
        ora.step(env.op.cpu().numpy(), env.mach.cpu().numpy())
    dense = ora.dense_adj()
    eq(env.dense_adj(torch.float64).cpu().numpy(), dense)
    eq(env.dense_adj(torch.float32).cpu().numpy(), dense.astype(np.float32))
    raw = env.raw_adj().cpu().numpy()[0]
    arc = dense[0].T != 0                                   # [u, v]
    np.fill_diagonal(arc, False)
    eq(np.diagonal(raw), 0)
    assert not (raw != 0)[~arc].any()                       # no weight where the observation has no arc
    mach = ora.export_state()["mach"][0]
    dur = np.where(mach >= 0, d["t"][0, np.arange(N), np.maximum(mach, 0)], 0.0)
    u, v = np.nonzero(arc)
    assert len(u) > N - J                                   # every job arc, and the machine arcs of the scheduled half
    sch = mach[u] >= 0
    assert (raw[u[~sch], v[~sch]] == 1).all()
    assert (raw[u[sch], v[sch]] >= np.trunc(dur[u[sch]])).all()   # so only a weight below 1 truncates to 0


# ---------------------------------------------------------------------------------------------------------------------
# packed host records
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("size", [(1678, 2, 1, 3), (48, 64, 4, 3), (1, 64, 8, 5), (1, 2, 1, 2)])
def test_packed_host_records_at_the_edges(size, pinned, monkeypatch):
    """Records of ~2 KB (J = 1678: 210 mask bytes), J = 48 at M = 64, and J = 1: the decoded records equal the
    device-pointer step, the padding is zero, and canary rows behind the batch stay untouched; with pinned buffers
    (the generic kernel writes the records straight into the mapped host buffer) and with pageable ones (staged copy)."""
    torch = _torch()
    monkeypatch.delenv("MTFJSP_HOST_ZEROCOPY", raising=False)
    pin = (lambda x: x.pin_memory()) if pinned else (lambda x: x)
    J, M, E, B = size
    N = J * M
    envm = _envm()
    d = ins.reference_stream_instances(B, J, M, E, 17)
    w = ins.random_weights(0, B, 17)
    envs = []
    for _ in range(2):
        env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32)
        env.load(d["t"], d["p"], d["transT"], d["edge"])
        env.scaler_init()
        env.reset(w)
        envs.append(env)
    dev_env, pk_env = envs
    nbytes = int(pk_env.host_buffers()[1].shape[1])
    used = 41 + (J + 7) // 8 + J
    assert nbytes == (used + 7) // 8 * 8
    pk_act = pin(torch.zeros((B, 2), dtype=torch.int32))
    guard = pin(torch.full((B + 4, nbytes), 0x5A, dtype=torch.uint8))   # four records of canary behind the batch
    pk_rec = guard[:B]
    check_obs = set(_checkpoints(N))
    for s in range(N):
        op, mach = dev_env.policy_random(seed=4)
        dev_env.step_obs(op, mach)
        pk_act[:, 0].copy_(op.cpu()); pk_act[:, 1].copy_(mach.cpu())
        pk_env.step_host_packed(pk_act, pk_rec)
        info6, cand, mask = pk_env.decode_records(pk_rec)
        tag = "step %d" % s
        eq(info6[:, 0], dev_env.reward5[:, 0].cpu().numpy(), err_msg=tag)
        eq(info6[:, 1], dev_env.done.cpu().numpy().astype(np.float64), err_msg=tag)
        eq(info6[:, 2:], dev_env.scaled4.cpu().numpy(), err_msg=tag)
        eq(cand, dev_env.candidate.cpu().numpy(), err_msg=tag)
        eq(mask, dev_env.job_mask.cpu().numpy(), err_msg=tag)
        raw = pk_rec.numpy()
        assert not raw[:, used:].any(), tag
        if J % 8:   # the unused bits of the last mask byte are zero too
            assert not (raw[:, 41 + (J - 1) // 8] >> (J % 8)).any(), tag
        assert bool((guard[B:] == 0x5A).all()), tag
        if s in check_obs:
            for name in ("task_fea", "mach_fea", "adj_w", "adj_src"):
                assert torch.equal(getattr(pk_env, name), getattr(dev_env, name)), (name, s)
    assert bool(dev_env.done.all())
    eq(pk_env.costs().cpu().numpy(), dev_env.costs().cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# device instance generator
# ---------------------------------------------------------------------------------------------------------------------

_U = np.uint64


def _splitmix64(x):
    x = x + _U(0x9E3779B97F4A7C15)
    x = (x ^ (x >> _U(30))) * _U(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> _U(27))) * _U(0x94D049BB133111EB)
    return x ^ (x >> _U(31))


def _u01(seed, env, item, k):
    """csrc/mtfjsp_env.cu u01: 53 bits of splitmix64(seed ^ splitmix64(env * c0 + item * c1 + k * c2)) -> [0, 1)."""
    env, item, k = (np.asarray(a, dtype=_U) for a in (env, item, k))
    with np.errstate(over="ignore"):
        inner = env * _U(0x100000001B3) + item * _U(0x9E3779B97F4A7C15) + k * _U(0xD1B54A32D192ED03)
        x = _splitmix64(_U(seed) ^ _splitmix64(inner))
    return (x >> _U(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def _generate_like_the_kernel(B, J, M, E, seed, env_offset):
    """instance_gen_kernel restated in numpy.  The kernel's file is compiled without FMA contraction, so every product
    and sum rounds on its own, as here: the values must agree exactly."""
    N = J * M
    env = (np.uint64(env_offset) + np.arange(B, dtype=_U))[:, None]          # [B, 1]
    op = np.arange(N, dtype=_U)[None, :]                                      # [1, N]
    avg_t = 1.0 + 98.0 * _u01(seed, env, op, 0)
    avg_p = 1.0 + 19.0 * _u01(seed, env, op, 1)
    k = np.minimum((_u01(seed, env, op, 2) * M).astype(np.int64), M - 1)      # [B, N] infeasible machines
    perm = np.broadcast_to(np.arange(M), (B, N, M)).copy()
    neg = np.zeros((B, N, M), dtype=bool)
    bi, ni = np.meshgrid(np.arange(B), np.arange(N), indexing="ij")
    for q in range(M - 1):                                                    # partial Fisher-Yates, k swaps per op
        act = q < k
        r = np.minimum(q + (_u01(seed, env, op, 3 + q) * (M - q)).astype(np.int64), M - 1)
        a, c = perm[:, :, q].copy(), perm[bi, ni, r]
        perm[:, :, q] = np.where(act, c, a)
        perm[bi, ni, r] = np.where(act, a, perm[bi, ni, r])
        sel = perm[:, :, q]
        neg[bi[act], ni[act], sel[act]] = True
    m = np.arange(M, dtype=_U)[None, None, :]
    tv = avg_t[:, :, None] * (0.8 + 0.4 * _u01(seed, env[:, :, None], op[:, :, None], _U(100) + m))
    pv = avg_p[:, :, None] * (0.8 + 0.4 * _u01(seed, env[:, :, None], op[:, :, None], _U(200) + m))
    t = np.where(neg, -tv, tv)
    p = np.where(neg, -pv, pv)
    avg = M // E
    grp = np.minimum(np.arange(M) // max(avg, 1), E - 1)
    lo, hi = np.triu_indices(M, k=1)
    dg = np.abs(grp[lo] - grp[hi]).astype(np.float64)
    u = _u01(seed, env, np.uint64(N) + (lo * M + hi).astype(_U)[None, :], 0)  # [B, pairs]
    v = np.where(dg == 0, 1.0 + 9.0 * u, 10.0 * dg + 10.0 * dg * u)
    tt = np.zeros((B, M, M))
    tt[:, lo, hi] = v
    tt[:, hi, lo] = v
    return dict(t=t, p=p, transT=tt, neg=neg, k=k)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(64, 64, 1), (64, 64, 7), (64, 64, 64), (5, 3, 2)])
def test_device_generator_equals_its_restatement(size):
    """mtfjsp_generate_instances at M = 64 (64-bit infeasibility masks, up to 63 Fisher-Yates swaps per op) with one
    group, ragged groups and one group per machine, and at a small M: every array equals the numpy restatement."""
    J, M, E = size
    B, first, seed = 3, 1000, 0xC0FFEE1234567890
    d = ins.device_instances(first, B, J, M, E, seed=seed)
    t, p, tt, edge = (d[k].cpu().numpy() for k in ("t", "p", "transT", "edge"))
    want = _generate_like_the_kernel(B, J, M, E, seed, first)
    eq(t < 0, want["neg"])                                  # sign pattern
    eq((t < 0).sum(-1), want["k"])                          # and count of infeasible machines
    if M == 64:   # the draw reaches the machines above bit 31 and the largest count
        assert want["k"].max() == M - 1 and want["neg"][:, :, 32:].any()
    eq(t, want["t"])
    eq(p, want["p"])
    eq(tt, want["transT"])
    eq(tt, np.transpose(tt, (0, 2, 1)))
    eq(np.diagonal(tt, axis1=1, axis2=2), 0.0)
    eg = ins.edge_groups(M, E)
    eq(edge, np.broadcast_to(eg, (B,) + eg.shape))
    gid = ins.edge_of_machine(eg, M)
    dist = np.abs(gid[:, None] - gid[None, :])
    off = ~np.eye(M, dtype=bool)
    lo = np.where(dist == 0, 1.0, 10.0 * dist); hi = np.where(dist == 0, 10.0, 20.0 * dist)
    assert (tt[:, off] >= lo[off]).all() and (tt[:, off] < hi[off]).all()   # transport-group distances
    part = ins.device_instances(first + 1, 1, J, M, E, seed=seed)
    eq(part["t"].cpu().numpy(), t[1:2])


@pytest.mark.gpu
def test_device_generator_needs_j_at_least_m():
    lib = _libm()
    with pytest.raises(lib.MTFJSPError, match=r"\(-1\).*J >= M"):
        ins.device_instances(0, 2, 63, 64, 4, seed=1)
    with pytest.raises(lib.MTFJSPError, match=r"\(-1\)"):
        ins.device_instances(0, 2, 1, 2, 1, seed=1)
    ins.device_instances(0, 2, 2, 2, 1, seed=1)             # J = M is the smallest it makes
