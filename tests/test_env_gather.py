"""mtfjsp_gather / BatchedMTFJSPEnv.gather_from: env b of one handle becomes a copy of env idx[b] of another.  After the
copy, every call on the destination must return the same bits as on a fresh env that replayed the source env's whole
history: checked here after every later step (observation rows, ELL adjacency, masks in both modes, candidates, actions
drawn from the masks, candidate-machine features, rewards, scaled rewards, done, costs, export_state, export_scaler),
across an episode boundary and into a second episode, at specialised, COLD and unspecialised sizes, with and without
left shift, under each environment switch, and around recorded (not yet performed) resets.  Rejected handle pairs leave
the destination as it was."""
import ctypes as C
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")
libm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200._lib")

E_ARG, E_STATE = -1, -3
SRC_B, DST_B = 7, 11
# idx: duplicates (3 three times, 0 twice), a permutation of 0..6 inside it, dst.B != src.B
IDX = np.array([3, 0, 6, 5, 3, 1, 2, 4, 0, 3, 6], dtype=np.int32)
OUT = ["op", "mach", "mfea1_buf", "mach_mask", "reward5", "scaled4", "done", "invalid", "task_fea", "mach_fea", "adj_w",
       "adj_src", "job_mask", "candidate"]


def _snap(env, with_outputs=True, state=True):
    out = {n: getattr(env, n).cpu().numpy().copy() for n in OUT} if with_outputs else {}
    if not state:
        return out
    out.update({"st_" + k: v.cpu().numpy() for k, v in env.export_state().items()})
    out.update({"sc_" + k: v.cpu().numpy() for k, v in env.export_scaler().items()})
    out["costs"] = env.costs().cpu().numpy()
    return out


def _same(a, b, where):
    assert a.keys() == b.keys()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg="%s: %s" % (where, k))


def _make(B, J, M, E, left_shift, d, w):
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=left_shift, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(w)
    env.obs(envm.MASK_ESA)
    return env


def _sub(d, idx):
    return {k: np.asarray(d[k])[idx] for k in ("t", "p", "transT", "edge")}


def _compare_step(dst, rep, where, seed, off=0, s=1):
    """One random step on both (the draw comes from each env's own masks), then every output.  Every second step (odd s)
    also the exported state and, every fourth, the other mask form: the other steps follow a step launch with nothing
    but reads of the outputs in between, so that they start overlapped (MTFJSP_LAUNCH_OVERLAP) where the size allows."""
    dst.random_step(seed=seed, env_offset=off)
    rep.random_step(seed=seed, env_offset=off)
    _same(_snap(dst, state=s % 2 == 1), _snap(rep, state=s % 2 == 1), where)
    if s % 4 != 3:
        return
    for env in (dst, rep):  # the other mask form, then back to the rollout's
        env.obs(envm.MASK_FINISHED)
    np.testing.assert_array_equal(dst.job_mask.cpu().numpy(), rep.job_mask.cpu().numpy(), err_msg=where + ": finished mask")
    np.testing.assert_array_equal(dst.candidate.cpu().numpy(), rep.candidate.cpu().numpy(), err_msg=where)
    for env in (dst, rep):
        env.obs(envm.MASK_ESA)


def _gather_vs_replay(J, M, E, left_shift, k, second=None):
    """src steps k times, dst (busy with other instances and a recorded reset) gathers IDX from it; then dst and a fresh
    replay env of the same prefixes finish the episode, reset (scaler carried over) and run `second` steps."""
    N = J * M
    second = min(N, 8) if second is None else second
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 1000 + J * M + k)
    w1 = ins.random_weights(0, SRC_B, 5)
    src = _make(SRC_B, J, M, E, left_shift, d, w1)
    acts = []
    for _ in range(k):
        src.random_step(seed=9, env_offset=3)
        acts.append((src.op.clone(), src.mach.clone()))
    d_other = ins.synthetic_instances(0, DST_B, J, M, E, 77)
    dst = _make(DST_B, J, M, E, left_shift, d_other, ins.random_weights(0, DST_B, 6))
    for _ in range(min(3, N)):
        dst.random_step(seed=1)
    idx = torch.as_tensor(IDX, device="cuda")
    dst.gather_from(src, idx)
    rep = _make(DST_B, J, M, E, left_shift, _sub(d, IDX), w1[IDX])
    for op, mach in acts:
        rep.step_obs(op[idx.long()], mach[idx.long()])
    _same(_snap(dst, with_outputs=False), _snap(rep, with_outputs=False), "right after the gather, k=%d" % k)
    for name in ("task_fea", "mach_fea", "adj_w", "adj_src", "job_mask", "candidate") + (("done", "invalid") if k else ()):
        np.testing.assert_array_equal(getattr(dst, name).cpu().numpy(), getattr(rep, name).cpu().numpy(), err_msg=name)
    for s in range(N - k):
        _compare_step(dst, rep, "episode 1, step %d of %d (k=%d)" % (k + s, N, k), seed=21, s=s)
    assert dst.done.cpu().numpy().all()
    w2 = torch.as_tensor(ins.random_weights(0, DST_B, 8), device="cuda")
    dst.reset(w2)  # recorded: the next random step performs it where the size's kernel can
    rep.reset(w2)
    for s in range(second):
        _compare_step(dst, rep, "episode 2, step %d (k=%d)" % (s, k), seed=22, off=5, s=s)
    return dst, rep


SIZES = [(6, 6, 2), (10, 10, 3), (30, 20, 5), (13, 11, 3)]  # specialised (fused reset, overlap), spec, COLD, generic


@pytest.mark.gpu
@pytest.mark.parametrize("left_shift", [True, False])
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%dE%d" % s)
def test_gather_equals_replay(size, left_shift):
    J, M, E = size
    N = J * M
    for k in sorted({0, 1, N // 2, N - 1, N}):
        _gather_vs_replay(J, M, E, left_shift, k, second=None if N <= 100 else 4)


@pytest.mark.gpu
@pytest.mark.parametrize("value", ["0", "1"])
@pytest.mark.parametrize("switch", ["MTFJSP_OBS_INCREMENTAL", "MTFJSP_LAUNCH_OVERLAP", "MTFJSP_FUSED_RESET",
                                    "MTFJSP_FORCE_GENERIC"])
@pytest.mark.parametrize("size", [(6, 6, 2), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_gather_equals_replay_under_switches(size, switch, value, monkeypatch):
    monkeypatch.setenv(switch, value)
    J, M, E = size
    _gather_vs_replay(J, M, E, True, (J * M) // 2)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"])
def test_gather_around_recorded_resets(fused, monkeypatch):
    """A reset (and scaler reset) recorded on src belongs to the copied state; one recorded on dst must not be performed
    on the copy by dst's next step; a reset of dst after a gather returns to the copied instance's reset image."""
    monkeypatch.setenv("MTFJSP_FUSED_RESET", fused)
    J, M, E = 6, 6, 2
    N = J * M
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 404)
    w1, w2 = ins.random_weights(0, SRC_B, 1), ins.random_weights(0, SRC_B, 2)
    idx = torch.as_tensor(IDX, device="cuda")
    # (a) src with a recorded reset + scaler reset after a finished episode
    src = _make(SRC_B, J, M, E, True, d, w1)
    acts = []
    for _ in range(N):
        src.random_step(seed=4)
        acts.append((src.op.clone(), src.mach.clone()))
    w2_src = torch.as_tensor(w2, device="cuda")
    src.reset(w2_src)
    src.scaler_reset()
    dst = _make(DST_B, J, M, E, True, ins.synthetic_instances(0, DST_B, J, M, E, 5), ins.random_weights(0, DST_B, 3))
    dst.gather_from(src, idx)
    rep = _make(DST_B, J, M, E, True, _sub(d, IDX), w1[IDX])
    for op, mach in acts:
        rep.step_obs(op[idx.long()], mach[idx.long()])
    rep.reset(w2[IDX])
    rep.scaler_reset()
    rep.obs(envm.MASK_ESA)
    dst.obs(envm.MASK_ESA)
    _same(_snap(dst, False), _snap(rep, False), "after gathering a recorded reset")
    for s in range(5):
        _compare_step(dst, rep, "after a recorded src reset, step %d" % s, seed=6, s=s)
    # (b) a reset recorded on dst, then a gather of a mid-episode src
    src2 = _make(SRC_B, J, M, E, True, d, w1)
    acts = []
    for _ in range(N // 2):
        src2.random_step(seed=8)
        acts.append((src2.op.clone(), src2.mach.clone()))
    w3 = torch.as_tensor(ins.random_weights(0, DST_B, 9), device="cuda")
    dst.reset(w3)  # recorded (fused) or performed; either way the gather must replace it
    dst.gather_from(src2, idx)
    rep2 = _make(DST_B, J, M, E, True, _sub(d, IDX), w1[IDX])
    for op, mach in acts:
        rep2.step_obs(op[idx.long()], mach[idx.long()])
    for s in range(3):
        _compare_step(dst, rep2, "after a recorded dst reset, step %d" % s, seed=10, s=s)
    # (c) reset of dst after the gather: the copied instances' reset image, the copied scaler carried over
    w4 = torch.as_tensor(ins.random_weights(0, DST_B, 11), device="cuda")
    dst.reset(w4)
    rep2.reset(w4)
    dst.obs(envm.MASK_ESA)
    rep2.obs(envm.MASK_ESA)
    _same(_snap(dst), _snap(rep2), "reset after the gather")
    fresh = _make(DST_B, J, M, E, True, _sub(d, IDX), w4)
    a, b = _snap(dst, False), _snap(fresh, False)
    for key in [k for k in a if k.startswith("st_")]:
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
    for name in ("task_fea", "adj_w", "adj_src", "job_mask", "candidate"):
        np.testing.assert_array_equal(getattr(dst, name).cpu().numpy(), getattr(fresh, name).cpu().numpy(), err_msg=name)
    for s in range(N):
        _compare_step(dst, rep2, "episode after the reset, step %d" % s, seed=12, s=s)


def test_gather_null_arguments_are_rejected_without_a_device():
    lib = libm.lib()
    assert lib.mtfjsp_gather(None, None, None, None) == E_ARG
    assert b"mtfjsp_gather" in lib.mtfjsp_last_error()
    assert lib.mtfjsp_bytes_per_gather(None) == 0


def _raw_gather(dst, src, idx):
    return dst._lib.mtfjsp_gather(dst._h, src._h, C.c_void_p(idx.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))


@pytest.mark.gpu
def test_rejected_handle_pairs_leave_dst_unchanged():
    J, M, E = 6, 6, 2
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 31)
    dd = ins.synthetic_instances(0, DST_B, J, M, E, 32)
    dst = _make(DST_B, J, M, E, True, dd, ins.random_weights(0, DST_B, 1))
    for _ in range(4):
        dst.random_step(seed=2)
    twin = _make(DST_B, J, M, E, True, dd, ins.random_weights(0, DST_B, 1))
    for _ in range(4):
        twin.random_step(seed=2)
    idx = torch.as_tensor(IDX, device="cuda")
    before = _snap(dst)

    def src_with(J_=J, M_=M, E_=E, ls=True, weights=(0.4, 0.4, 0.2), divisor=1.0, gamma=0.99, load=True):
        s = envm.BatchedMTFJSPEnv(SRC_B, J_, M_, E_, left_shift=ls, weights=weights, scaling_divisor=divisor, gamma=gamma,
                                  obs_dtype=torch.float32)
        if load:
            x = ins.synthetic_instances(0, SRC_B, J_, M_, E_, 33) if (J_, M_, E_) != (J, M, E) else d
            s.load(x["t"], x["p"], x["transT"], x["edge"])
            s.scaler_init()
            s.reset(ins.random_weights(0, SRC_B, 3))
        return s

    cases = [(dst, E_ARG), (src_with(J_=7), E_ARG), (src_with(M_=5, J_=7), E_ARG), (src_with(E_=3), E_ARG),
             (src_with(ls=False), E_ARG), (src_with(weights=(0.5, 0.3, 0.2)), E_ARG), (src_with(divisor=2.0), E_ARG),
             (src_with(gamma=0.9), E_ARG), (src_with(load=False), E_STATE)]
    for src, code in cases:
        assert _raw_gather(dst, src, idx) == code, libm.lib().mtfjsp_last_error()
        if src is not dst:
            with pytest.raises(libm.MTFJSPError):
                dst.gather_from(src, idx)
        _same(_snap(dst), before, "after a rejected gather")
    for s in range(5):  # the handle goes on exactly as an untouched twin
        _compare_step(dst, twin, "after rejected gathers, step %d" % s, seed=3, s=s)


@pytest.mark.gpu
def test_out_of_range_index_sets_only_the_invalid_flag():
    J, M, E = 6, 6, 2
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 41)
    src = _make(SRC_B, J, M, E, True, d, ins.random_weights(0, SRC_B, 1))
    for _ in range(10):
        src.random_step(seed=4)
    dd = ins.synthetic_instances(0, DST_B, J, M, E, 42)
    dst = _make(DST_B, J, M, E, True, dd, ins.random_weights(0, DST_B, 2))
    for _ in range(3):
        dst.random_step(seed=5)
    dst.invalid.zero_()
    before = _snap(dst)
    bad = np.array([1, 4, 9])
    raw = IDX.copy()
    raw[bad] = [-1, SRC_B, 1 << 30]
    dst.gather_from(src, torch.as_tensor(raw, device="cuda"))
    after = _snap(dst)
    good = np.setdiff1d(np.arange(DST_B), bad)
    ref = _snap(src)
    np.testing.assert_array_equal(after["invalid"], np.isin(np.arange(DST_B), bad).astype(np.uint8))
    for key in after:
        if key == "invalid":
            continue
        np.testing.assert_array_equal(after[key][bad], before[key][bad], err_msg="untouched: " + key)
        np.testing.assert_array_equal(after[key][good], ref[key][raw[good]], err_msg="gathered: " + key)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(6, 6, 2), (13, 11, 3)], ids=lambda s: "J%dM%dE%d" % s)
def test_raw_gather_breaks_the_incremental_observation_chain(size):
    """Through the bare C entry point the destination's observation buffers are not copied: they still hold dst's own
    previous observation.  dst's next step into those same buffers must therefore rewrite every row, not only the rows the
    step changes (obs_synced = false in mtfjsp_gather)."""
    J, M, E = size
    N = J * M
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 61)
    w1 = ins.random_weights(0, SRC_B, 61)
    src = _make(SRC_B, J, M, E, True, d, w1)
    acts = []
    for _ in range(N // 2):
        src.random_step(seed=7)
        acts.append((src.op.clone(), src.mach.clone()))
    dst = _make(DST_B, J, M, E, True, ins.synthetic_instances(0, DST_B, J, M, E, 62), ins.random_weights(0, DST_B, 62))
    for _ in range(3):  # dst's buffers become the incremental mirror of dst's own state
        dst.random_step(seed=2)
    idx = torch.as_tensor(IDX, device="cuda")
    assert _raw_gather(dst, src, idx) == 0
    rep = _make(DST_B, J, M, E, True, _sub(d, IDX), w1[IDX])
    for op, mach in acts:
        rep.step_obs(op[idx.long()], mach[idx.long()])
    for s in range(4):
        _compare_step(dst, rep, "after a raw gather, step %d" % s, seed=8, s=s)


@pytest.mark.gpu
def test_source_steps_on_after_a_gather():
    """The gather is a non-step call on the source too: src's next random steps (overlapped ones at J6M6) continue
    exactly as those of an untouched twin."""
    J, M, E = 6, 6, 2
    N = J * M
    d = ins.synthetic_instances(0, SRC_B, J, M, E, 71)
    w1 = ins.random_weights(0, SRC_B, 71)
    src, twin = _make(SRC_B, J, M, E, True, d, w1), _make(SRC_B, J, M, E, True, d, w1)
    for _ in range(5):
        src.random_step(seed=3)
        twin.random_step(seed=3)
    dst = _make(DST_B, J, M, E, True, ins.synthetic_instances(0, DST_B, J, M, E, 72), ins.random_weights(0, DST_B, 72))
    dst.gather_from(src, torch.as_tensor(IDX, device="cuda"))
    for s in range(N - 5):
        _compare_step(src, twin, "source after the gather, step %d" % s, seed=3, s=s)
