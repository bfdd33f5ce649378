"""The episode reset folded into the next step launch (MTFJSP_FUSED_RESET, default on) against the eager reset
(MTFJSP_FUSED_RESET=0: reset_copy_kernel + scaler_kernel at the call).  Every call sequence below must leave
bit-identical state (export_state, export_scaler, costs) and bit-identical outputs on both paths.  The sequences
cover the fused step, each entry point that runs a recorded reset before it reads the state, and seed, env offset
or mask mode changes between random steps."""
import importlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ins = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.instances")
envm = importlib.import_module("e2e-mappo-for-mt-fjsp_b200.env")

B = 37  # not a multiple of the envs per warp or block: idle groups in the last warp
SIZES = [(6, 6, 2), (10, 10, 3), (15, 10, 2)]  # (15, 10): COLD kernel, which runs the recorded reset before its step


def first_actions(d):
    """op 0 (job 0's first op, its candidate after a reset) on its first feasible machine"""
    t0 = np.asarray(d["t"])[:, 0, :]
    return (torch.zeros(B, dtype=torch.int32, device="cuda"),
            torch.as_tensor(np.argmax(t0 >= 0, axis=1).astype(np.int32), device="cuda"))


def outputs(env):
    names = ["op", "mach", "mfea1_buf", "mach_mask", "reward5", "scaled4", "done", "invalid", "task_fea", "mach_fea",
             "adj_w", "adj_src", "job_mask", "candidate"]
    return {n: getattr(env, n).cpu().numpy().copy() for n in names}


def state(env):
    out = {"st_" + k: v.cpu().numpy() for k, v in env.export_state().items()}
    out.update({"sc_" + k: v.cpu().numpy() for k, v in env.export_scaler().items()})
    out["costs"] = env.costs().cpu().numpy()
    return out


def run(size, seq, fused, monkeypatch):
    J, M, E = size
    monkeypatch.setenv("MTFJSP_FUSED_RESET", "1" if fused else "0")
    d = ins.synthetic_instances(0, B, J, M, E, 21)
    ctx = {"w1": torch.as_tensor(ins.random_weights(0, B, 21), device="cuda"),
           "w2": torch.as_tensor(ins.random_weights(0, B, 22), device="cuda"),
           "w3": torch.as_tensor(ins.random_weights(0, B, 23), device="cuda")}
    env = envm.BatchedMTFJSPEnv(B, J, M, E, left_shift=True, obs_dtype=torch.float32, mask_mode=envm.MASK_ESA)
    env.load(d["t"], d["p"], d["transT"], d["edge"])
    env.scaler_init()
    env.reset(ctx["w1"])  # the first reset takes the snapshot; the ones below are recorded (fused) or copied (eager)
    for s in range(5):  # mid-episode state, running scaler statistics that a reset must keep
        env.random_step(seed=3, env_offset=11)
    rec = []
    for op in seq:
        kind, arg = op if isinstance(op, tuple) else (op, None)
        if kind == "reset":
            env.reset(ctx[arg])
        elif kind == "scaler_reset":
            env.scaler_reset()
        elif kind == "random_step":
            seed, off, mm = arg if arg else (3, 11, None)
            env.random_step(seed=seed, env_offset=off, mask_mode=mm)
            rec.append(outputs(env))
        elif kind == "obs":
            env.obs()
            rec.append(outputs(env))
        elif kind == "step_obs":
            env.step_obs(*first_actions(d))
            rec.append(outputs(env))
        elif kind == "step_host_packed":
            acts = torch.stack([x.cpu() for x in first_actions(d)], 1).contiguous().pin_memory()
            recs = env.host_buffers()[1]
            env.step_host_packed(acts, recs)
            rec.append({"records": recs.numpy().copy(), **outputs(env)})
        elif kind == "costs":
            rec.append({"costs": env.costs().cpu().numpy()})
        elif kind == "export_state":
            rec.append(state(env))
        elif kind == "dense_adj":
            rec.append({"dense_adj": env.dense_adj().cpu().numpy()})
        else:
            raise ValueError(kind)
    for s in range(3):  # the episode goes on from whatever the sequence left
        env.random_step(seed=5, env_offset=11)
        rec.append(outputs(env))
    rec.append(state(env))
    torch.cuda.synchronize()
    return rec, env.launch_count


SEQUENCES = {
    "reset_step": ["reset", "random_step"],
    "reset_scaler_step": ["reset", "scaler_reset", "random_step"],
    "scaler_reset_then_reset": ["scaler_reset", "reset", "random_step"],
    "reset_twice_new_weights": ["reset", ("reset", "w3"), "random_step"],
    "reset_scaler_reset": ["reset", "scaler_reset", ("reset", "w3"), "random_step"],
    "reset_obs": ["reset", "scaler_reset", "obs", "random_step"],
    "reset_step_obs": ["reset", "scaler_reset", "step_obs", "random_step"],
    "reset_step_host_packed": ["reset", "scaler_reset", "step_host_packed", "random_step"],
    "reset_costs": ["reset", "scaler_reset", "costs", "random_step"],
    "reset_export_state": ["reset", "scaler_reset", "export_state", "random_step"],
    "reset_dense_adj": ["reset", "scaler_reset", "dense_adj", "random_step"],
    "seed_and_offset_change": ["reset", "random_step", ("random_step", (9, 11, None)), ("random_step", (9, 0, None)),
                               ("random_step", (3, 11, None))],
    "mask_mode_change": ["reset", ("random_step", (3, 11, envm.MASK_FINISHED)), ("random_step", (3, 11, envm.MASK_ESA)),
                         ("random_step", (3, 11, envm.MASK_FINISHED))],
}


@pytest.mark.parametrize("name", sorted(SEQUENCES))
@pytest.mark.parametrize("size", SIZES, ids=lambda s: "J%dM%d" % s[:2])
def test_fused_reset_matches_eager_reset(size, name, monkeypatch):
    seq = [("reset", "w2") if op == "reset" else op for op in SEQUENCES[name]]
    got, n_fused = run(size, seq, True, monkeypatch)
    want, n_eager = run(size, seq, False, monkeypatch)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.keys() == w.keys()
        for k in w:
            np.testing.assert_array_equal(g[k], w[k], err_msg="record %d, %s" % (i, k))
    if size[:2] in ((6, 6), (10, 10)) and seq[:2] == [("reset", "w2"), "random_step"]:
        assert n_fused == n_eager - 1  # the reset copy ran inside the step launch

