"""Device-resident batched MT-FJSP environment over the C ABI (include/mtfjsp.h).

`BatchedMTFJSPEnv` is the native interface: every input and output is a torch CUDA tensor, nothing
synchronises the host.  torch is plumbing here (device memory + streams); all environment arithmetic
happens in the sm_100a kernels of csrc/mtfjsp_env.cu.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check

F32, F64 = 0, 1
MASK_FINISHED, MASK_ESA = 0, 1


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _to_dev(x, device, dtype):
    if not torch.is_tensor(x):
        x = torch.as_tensor(np.ascontiguousarray(x))
    return x.to(device=device, dtype=dtype).contiguous()


def _on(device, *tensors):
    """Every tensor handed to the library must live on the handle's device (raw pointers cross the C ABI)."""
    for t in tensors:
        if t is not None and t.device != device:
            raise ValueError("tensor on %s passed to an environment on %s" % (t.device, device))


class BatchedMTFJSPEnv:
    """B environments of J jobs x M operations on M machines on one GPU.

    Mirrors the environment half of the reference's Parallel_env (trainer/parallel_env.py:19-282) plus the
    job-mask bookkeeping (algorithm/ppo_algorithm.py:202-317); see include/mtfjsp.h for the per-call
    reference locations."""

    def __init__(self, B, J, M, E, left_shift=True, weights=(0.4, 0.4, 0.2), scaling_divisor=1.0, gamma=0.99,
                 device=None, obs_dtype=torch.float32, mask_mode=MASK_ESA, incremental_obs=True):
        """incremental_obs: fused steps rewrite only the observation rows a step changes (the object owns
        task_fea / mach_fea / adj_w / adj_src; callers read them, or copy them, and never write into them)."""
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedMTFJSPEnv needs a CUDA device (there is no CPU fallback)")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedMTFJSPEnv needs a CUDA device (there is no CPU fallback)")
        if self.device.index is None:  # "cuda" without an index means the CURRENT device, not device 0
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.B, self.J, self.M, self.E, self.N = B, J, M, E, J * M
        self.obs_dtype = obs_dtype
        self._dt = F64 if obs_dtype == torch.float64 else F32
        self.mask_mode = mask_mode
        self._lib = _lib.lib()
        h = C.c_void_p()
        check(self._lib.mtfjsp_create(C.byref(h), B, J, M, E, int(bool(left_shift)), self.device.index), "mtfjsp_create")
        self._h = h
        check(self._lib.mtfjsp_set_params(self._h, weights[0], weights[1], weights[2], scaling_divisor, gamma), "mtfjsp_set_params")
        check(self._lib.mtfjsp_set_obs_incremental(self._h, int(bool(incremental_obs))), "mtfjsp_set_obs_incremental")
        dev, N = self.device, self.N
        self.task_fea = torch.empty((B, N, 12), dtype=obs_dtype, device=dev)
        self.mach_fea = torch.empty((B, M, 8), dtype=obs_dtype, device=dev)
        self.adj_w = torch.empty((B, N, 2), dtype=torch.float32, device=dev)
        self.adj_src = torch.empty((B, N), dtype=torch.int16, device=dev)
        self.job_mask = torch.empty((B, J), dtype=torch.uint8, device=dev)
        self.candidate = torch.empty((B, J), dtype=torch.int32, device=dev)
        self.reward5 = torch.empty((B, 5), dtype=torch.float64, device=dev)
        self.scaled4 = torch.empty((B, 4), dtype=torch.float64, device=dev)
        self.done = torch.empty((B,), dtype=torch.uint8, device=dev)
        self.invalid = torch.empty((B,), dtype=torch.uint8, device=dev)
        self.mfea1_buf = torch.empty((B, M, 6), dtype=obs_dtype, device=dev)
        self.mach_mask = torch.empty((B, M), dtype=torch.uint8, device=dev)
        self.op = torch.empty((B,), dtype=torch.int32, device=dev)
        self.mach = torch.empty((B,), dtype=torch.int32, device=dev)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.mtfjsp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- instance data -------------------------------------------------------------------------------------
    def load(self, t, p, tt, edge):
        """t, p [B,N,M]; tt [B,M,M]; edge [B,E,W] machine ids padded with -1 (numpy or torch)."""
        dev = self.device
        t = _to_dev(t, dev, torch.float64)
        p = _to_dev(p, dev, torch.float64)
        tt = _to_dev(tt, dev, torch.float64)
        edge = _to_dev(edge, dev, torch.int32)
        assert t.shape == (self.B, self.N, self.M) and p.shape == t.shape and tt.shape == (self.B, self.M, self.M)
        assert edge.dim() == 3 and tuple(edge.shape[:2]) == (self.B, self.E)
        check(self._lib.mtfjsp_load(self._h, _ptr(t), _ptr(p), _ptr(tt), _ptr(edge), edge.shape[2], _stream()), "mtfjsp_load")
        self._keep = (t, p, tt, edge)  # the library copies on the stream; keep the sources alive until then

    def scaler_init(self):
        check(self._lib.mtfjsp_scaler_init(self._h, _stream()), "mtfjsp_scaler_init")

    def scaler_reset(self):
        check(self._lib.mtfjsp_scaler_reset(self._h, _stream()), "mtfjsp_scaler_reset")

    def reset(self, weights):
        w = _to_dev(weights, self.device, torch.float64)
        assert tuple(w.shape) == (self.B, 3)
        check(self._lib.mtfjsp_reset(self._h, _ptr(w), _stream()), "mtfjsp_reset")
        self._w = w

    # ---- hot path ----------------------------------------------------------------------------------------------
    def step(self, op, mach):
        _on(self.device, op, mach)
        check(self._lib.mtfjsp_step(self._h, _ptr(op), _ptr(mach), _ptr(self.reward5), _ptr(self.scaled4),
                                    _ptr(self.done), _ptr(self.invalid), _stream()), "mtfjsp_step")
        return self.reward5, self.scaled4, self.done, self.invalid

    def obs(self, mask_mode=None):
        mm = self.mask_mode if mask_mode is None else mask_mode
        check(self._lib.mtfjsp_obs(self._h, _ptr(self.task_fea), _ptr(self.mach_fea), _ptr(self.adj_w), _ptr(self.adj_src),
                                   _ptr(self.job_mask), _ptr(self.candidate), mm, self._dt, _stream()), "mtfjsp_obs")
        return self.task_fea, self.mach_fea, self.adj_w, self.adj_src, self.job_mask, self.candidate

    def step_obs(self, op, mach, mask_mode=None):
        mm = self.mask_mode if mask_mode is None else mask_mode
        _on(self.device, op, mach)
        check(self._lib.mtfjsp_step_obs(self._h, _ptr(op), _ptr(mach), _ptr(self.reward5), _ptr(self.scaled4),
                                        _ptr(self.done), _ptr(self.invalid), _ptr(self.task_fea), _ptr(self.mach_fea),
                                        _ptr(self.adj_w), _ptr(self.adj_src), _ptr(self.job_mask), _ptr(self.candidate),
                                        mm, self._dt, _stream()), "mtfjsp_step_obs")

    def mfea1(self, op):
        _on(self.device, op)
        check(self._lib.mtfjsp_mfea1(self._h, _ptr(op), _ptr(self.mfea1_buf), _ptr(self.mach_mask), self._dt, _stream()),
              "mtfjsp_mfea1")
        return self.mfea1_buf, self.mach_mask

    def policy_random(self, seed, env_offset=0, mask_mode=None):
        mm = self.mask_mode if mask_mode is None else mask_mode
        check(self._lib.mtfjsp_policy_random(self._h, seed, env_offset, mm, _ptr(self.op), _ptr(self.mach), _stream()),
              "mtfjsp_policy_random")
        return self.op, self.mach

    def random_step(self, seed, env_offset=0, mask_mode=None, with_mfea1=True):
        """policy_random -> mfea1 -> step_obs: the environment side of one rollout step."""
        mm = self.mask_mode if mask_mode is None else mask_mode
        check(self._lib.mtfjsp_random_step(
            self._h, seed, env_offset, _ptr(self.op), _ptr(self.mach), _ptr(self.mfea1_buf) if with_mfea1 else None,
            _ptr(self.mach_mask) if with_mfea1 else None, _ptr(self.reward5), _ptr(self.scaled4), _ptr(self.done),
            _ptr(self.invalid), _ptr(self.task_fea), _ptr(self.mach_fea), _ptr(self.adj_w), _ptr(self.adj_src),
            _ptr(self.job_mask), _ptr(self.candidate), mm, self._dt, _stream()), "mtfjsp_random_step")

    def step_host(self, op_host, mach_host, info6_host, job_mask_host, candidate_host, mask_mode=None):
        """Host-buffer step (pinned int32 / float64 / uint8 / int32 torch CPU tensors); obs stay on device."""
        mm = self.mask_mode if mask_mode is None else mask_mode
        check(self._lib.mtfjsp_step_host(self._h, _ptr(op_host), _ptr(mach_host), _ptr(info6_host), _ptr(job_mask_host),
                                         _ptr(candidate_host), _ptr(self.task_fea), _ptr(self.mach_fea), _ptr(self.adj_w),
                                         _ptr(self.adj_src), mm, self._dt, _stream()), "mtfjsp_step_host")

    def host_record_dtype(self):
        """numpy structured dtype of one packed host-step record (include/mtfjsp.h: mtfjsp_step_host_packed):
        r, scaled4 = (mk_s, idle_s, pt_s, tt_s), done, mask_bits (bit j & 7 of byte j >> 3: job j not selectable),
        next_op (candidate op of job j = j * M + next_op[j])."""
        nbytes = int(self._lib.mtfjsp_host_record_bytes(self._h))
        mb = (self.J + 7) // 8
        return np.dtype({"names": ["r", "scaled4", "done", "mask_bits", "next_op"],
                         "formats": ["<f8", ("<f8", 4), "u1", ("u1", mb), ("u1", self.J)],
                         "offsets": [0, 8, 40, 41, 41 + mb], "itemsize": nbytes})

    def decode_records(self, records_host):
        """Packed host-step records -> the arrays of the split call: info6 [B,6] f64 = (r, done, mk_s, idle_s, pt_s, tt_s)
        (trainer/parallel_env.py:260), candidate [B,J] int32, job_mask [B,J] uint8."""
        rec = records_host.numpy() if isinstance(records_host, torch.Tensor) else np.asarray(records_host)
        rec = rec.view(self.host_record_dtype())[:, 0]
        info6 = np.empty((rec.shape[0], 6), dtype=np.float64)
        info6[:, 0] = rec["r"]; info6[:, 1] = rec["done"]; info6[:, 2:] = rec["scaled4"]
        candidate = np.arange(self.J, dtype=np.int32)[None, :] * self.M + rec["next_op"].astype(np.int32)
        job_mask = np.unpackbits(rec["mask_bits"], axis=1, bitorder="little")[:, :self.J]
        return info6, candidate, job_mask

    def host_buffers(self):
        """Pinned host buffers for step_host_packed: actions [B,2] int32 and records [B, record_bytes] uint8
        (view the latter with `.numpy().view(env.host_record_dtype())[:, 0]`)."""
        nbytes = int(self._lib.mtfjsp_host_record_bytes(self._h))
        return (torch.zeros((self.B, 2), dtype=torch.int32).pin_memory(),
                torch.zeros((self.B, nbytes), dtype=torch.uint8).pin_memory())

    def step_host_packed(self, actions_host, records_host, mask_mode=None):
        """Host-buffer step, one copy each way: actions_host [B,2] int32 (op, machine) pairs in, packed step records
        out (info6, candidates, job mask per env); observations stay on the device."""
        mm = self.mask_mode if mask_mode is None else mask_mode
        check(self._lib.mtfjsp_step_host_packed(self._h, _ptr(actions_host), _ptr(records_host), _ptr(self.task_fea),
                                                _ptr(self.mach_fea), _ptr(self.adj_w), _ptr(self.adj_src), mm, self._dt,
                                                _stream()), "mtfjsp_step_host_packed")

    def host_stepper(self, records_host, mask_mode=None):
        """Prepared form of step_host_packed for a host loop that reuses its buffers: binds everything that does not
        change between steps once and returns `step(actions_ptr)`, where actions_ptr is the address (int) of a pinned
        [B,2] int32 action array, e.g. `acts[s].data_ptr()`.  Saves the per-call argument marshalling (6 pointer
        objects, stream lookup by attribute chain) of the general method -- a few microseconds of a ~170 us step."""
        mm = self.mask_mode if mask_mode is None else mask_mode
        fn, h = self._lib.mtfjsp_step_host_packed, self._h
        rec, tf, mf, aw, asrc = (_ptr(x) for x in (records_host, self.task_fea, self.mach_fea, self.adj_w, self.adj_src))
        dt = self._dt
        keep = records_host  # the closure keeps the record buffer alive
        cur = torch.cuda.current_stream

        def step(actions_ptr):
            rc = fn(h, actions_ptr, rec, tf, mf, aw, asrc, mm, dt, cur().cuda_stream)
            if rc:
                check(rc, "mtfjsp_step_host_packed")
            return keep

        return step

    # buffers this class owns and hands to the library: what gather_from copies besides the handle's own state
    _OWNED = ("task_fea", "mach_fea", "adj_w", "adj_src", "job_mask", "candidate", "reward5", "scaled4", "done", "invalid",
              "op", "mach", "mfea1_buf", "mach_mask")

    def gather_from(self, src, idx):
        """Env b of this object becomes a copy of env idx[b] of `src` (idx [B] integers; duplicates and permutations are
        allowed, src.B may differ).  The handle's state -- records, static tables, reset snapshot, masks, candidates,
        reward-scaler state -- goes through mtfjsp_gather; the buffers this object owns (observation, masks, candidates,
        step outputs, last actions, candidate-machine features) are copied by index on the device.  Afterwards the object
        is indistinguishable from one that stepped there itself.  An idx entry outside [0, src.B) leaves env b as it was
        and sets its invalid flag.  src and this object must have the same sizes, left_shift, reward parameters and
        observation dtype (MTFJSPError / ValueError otherwise); src must have been loaded."""
        if not isinstance(src, BatchedMTFJSPEnv):
            raise TypeError("gather_from needs a BatchedMTFJSPEnv")
        if src.obs_dtype != self.obs_dtype:
            raise ValueError("gather_from between environments of different observation dtypes")
        idx = _to_dev(idx, self.device, torch.int32)
        if tuple(idx.shape) != (self.B,):
            raise ValueError("idx must have shape [%d]" % self.B)
        check(self._lib.mtfjsp_gather(self._h, src._h, _ptr(idx), _stream()), "mtfjsp_gather")
        ok = (idx >= 0) & (idx < src.B)
        i = torch.where(ok, idx, 0).long()
        # two launches per buffer, written in place (the library tracks the observation pointers)
        for name in self._OWNED:
            d = getattr(self, name)
            if name == "invalid":
                torch.index_select(src.invalid, 0, i, out=d)
                d.masked_fill_(~ok, 1)
            else:
                torch.where(ok.view((-1,) + (1,) * (d.dim() - 1)), getattr(src, name).index_select(0, i), d, out=d)

    # ---- one-step lookahead ----------------------------------------------------------------------------------------
    def peek(self, op, mach):
        """What `step` would return for each of K (op, machine) pairs per env, without changing the env (mtfjsp_peek).
        op, mach: [B,K] integer tensors on this env's device.  Returns (reward5 [B,K,5] f64 = (r, r_mk, r_idle, r_pt,
        r_tt), bit for bit the step's; invalid [B,K] u8, the step's invalid flag, zeros in reward5 where set), in new
        buffers.  No scaled rewards: the reward scaler does not advance."""
        _on(self.device, op, mach)
        if op.dim() != 2 or op.shape[0] != self.B or tuple(mach.shape) != tuple(op.shape):
            raise ValueError("op and mach must both have shape [%d, K]" % self.B)
        op = op.to(torch.int32).contiguous()
        mach = mach.to(torch.int32).contiguous()
        K = op.shape[1]
        r5 = torch.empty((self.B, K, 5), dtype=torch.float64, device=self.device)
        inv = torch.empty((self.B, K), dtype=torch.uint8, device=self.device)
        check(self._lib.mtfjsp_peek(self._h, _ptr(op), _ptr(mach), K, _ptr(r5), _ptr(inv), _stream()), "mtfjsp_peek")
        return r5, inv

    def candidate_ops(self):
        """[B,J] int32: the next op of every job from the env's current schedule (j*M + the number of its scheduled ops,
        the job's last op once it is finished).  Read from the handle's state, so it is current after any call -- unlike
        the `candidate` buffer, which follows observation-writing steps only."""
        mach = torch.empty((self.B, self.N), dtype=torch.int32, device=self.device)
        check(self._lib.mtfjsp_export_state(self._h, _ptr(mach), None, None, None, _stream()), "mtfjsp_export_state")
        nx = (mach.view(self.B, self.J, self.M) >= 0).sum(dim=2, dtype=torch.int32)  # a job's scheduled ops are a prefix
        base = torch.arange(self.J, dtype=torch.int32, device=self.device) * self.M
        return base + torch.clamp(nx, max=self.M - 1)

    def peek_candidates(self, machines=None):
        """peek over the candidate op of every job.  machines=None: every (candidate op of job j, machine m) pair,
        returns reward5 [B,J,M,5] and invalid [B,J,M].  machines [B,N] integers (a machine for every op, as the machine
        rules produce): the pair (candidate op of job j, machines[b, op]), returns reward5 [B,J,5] and invalid [B,J].
        The candidate of a finished job is its last op, already scheduled: reported invalid."""
        B, J, M = self.B, self.J, self.M
        cand = self.candidate_ops()
        if machines is None:
            op = cand.unsqueeze(2).expand(B, J, M).reshape(B, J * M)
            mach = torch.arange(M, dtype=torch.int32, device=self.device).repeat(J).expand(B, J * M)
            r5, inv = self.peek(op, mach)
            return r5.view(B, J, M, 5), inv.view(B, J, M)
        _on(self.device, machines)
        if tuple(machines.shape) != (B, self.N):
            raise ValueError("machines must have shape [%d, %d]" % (B, self.N))
        return self.peek(cand, torch.gather(machines, 1, cand.long()))

    # ---- whole-episode replay ----------------------------------------------------------------------------------------
    def replay(self, actions, src=None):
        """What T steps of each of R action sequences leave, each from the episode start of env src[r], without changing
        the env (mtfjsp_replay).  actions: [T,R,2] integer (op, machine) tensor on this env's device, 1 <= T <= N -- the
        [N,S,2] layout greedy_validate, beam_validate and the rules' rollouts return.  src: [R] integers (duplicates and
        permutations allowed); None means arange(B) and needs R == B.  Returns new tensors final4 [R,4] f64 (what `costs`
        would return), return5 [R,5] f64 (the step-order sum of the steps' reward5) and first_invalid [R] int32 (-1, or the
        index of the first invalid action, which was a no-op; -2 where src is outside [0, B), with zero rows)."""
        _on(self.device, actions, src)
        if actions.dim() != 3 or actions.shape[2] != 2:
            raise ValueError("actions must have shape [T, R, 2]")
        T, R = int(actions.shape[0]), int(actions.shape[1])
        if src is None:
            if R != self.B:
                raise ValueError("src=None replays env r from row r: needs R == B = %d" % self.B)
            src = torch.arange(R, dtype=torch.int32, device=self.device)
        elif tuple(src.shape) != (R,):
            raise ValueError("src must have shape [%d]" % R)
        src = src.to(torch.int32).contiguous()
        act = actions.to(torch.int32).transpose(0, 1).contiguous()  # [R,T,2]: one contiguous run per candidate
        final4 = torch.empty((R, 4), dtype=torch.float64, device=self.device)
        ret5 = torch.empty((R, 5), dtype=torch.float64, device=self.device)
        finv = torch.empty((R,), dtype=torch.int32, device=self.device)
        check(self._lib.mtfjsp_replay(self._h, _ptr(src), R, _ptr(act), T, _ptr(final4), _ptr(ret5), _ptr(finv),
                                      _stream()), "mtfjsp_replay")
        return final4, ret5, finv

    # ---- views ---------------------------------------------------------------------------------------------------
    def dense_adj(self, dtype=torch.float64):
        adj = torch.empty((self.B, self.N, self.N), dtype=dtype, device=self.device)
        check(self._lib.mtfjsp_dense_adj(self._h, _ptr(adj), F64 if dtype == torch.float64 else F32, _stream()), "mtfjsp_dense_adj")
        return adj

    def raw_adj(self):
        """int32 [B,N,N], adj[b,u,v] = trunc(weight of arc u -> v): the reference's nx.to_numpy_array(G)[1:-1,1:-1].astype(int)."""
        adj = torch.empty((self.B, self.N, self.N), dtype=torch.int32, device=self.device)
        check(self._lib.mtfjsp_raw_adj(self._h, _ptr(adj), _stream()), "mtfjsp_raw_adj")
        return adj

    def costs(self, with_total_e1=False):
        c = torch.empty((self.B, 4), dtype=torch.float64, device=self.device)
        e1 = torch.empty((self.B,), dtype=torch.float64, device=self.device) if with_total_e1 else None
        check(self._lib.mtfjsp_costs(self._h, _ptr(c), _ptr(e1), _stream()), "mtfjsp_costs")
        return (c, e1) if with_total_e1 else c

    def export_state(self):
        dev, B, N, M = self.device, self.B, self.N, self.M
        mach = torch.empty((B, N), dtype=torch.int32, device=dev)
        st = torch.empty((B, N), dtype=torch.float64, device=dev)
        ft = torch.empty((B, N), dtype=torch.float64, device=dev)
        routes = torch.empty((B, M, N), dtype=torch.int32, device=dev)
        check(self._lib.mtfjsp_export_state(self._h, _ptr(mach), _ptr(st), _ptr(ft), _ptr(routes), _stream()), "mtfjsp_export_state")
        return dict(mach=mach, st=st, ft=ft, routes=routes)

    def export_scaler(self):
        dev, B = self.device, self.B
        R = torch.empty((B, 4), dtype=torch.float64, device=dev)
        mean = torch.empty_like(R)
        S = torch.empty_like(R)
        n = torch.empty((B,), dtype=torch.int64, device=dev)
        check(self._lib.mtfjsp_export_scaler(self._h, _ptr(R), _ptr(mean), _ptr(S), _ptr(n), _stream()), "mtfjsp_export_scaler")
        return dict(R=R, mean=mean, S=S, n=n)

    @property
    def launch_count(self):
        return int(self._lib.mtfjsp_launch_count(self._h))

    @property
    def launch_overlap_error(self):
        """Nonzero if an overlapped step launch timed out waiting for its predecessor (every later call raises)."""
        return int(self._lib.mtfjsp_launch_overlap_error(self._h))

    def check_launch_overlap(self):
        """Raises if a step launch timed out waiting for its predecessor and went on with what it found.  Call it after
        synchronising with the device: the word is final for every launch that has finished."""
        if self.launch_overlap_error:
            raise _lib.MTFJSPError("a step launch waited more than 1 s for the previous one (launch overlap): "
                                   "its results are not trustworthy")

    def bytes_per_step(self):
        return int(self._lib.mtfjsp_bytes_per_step(self._h, self._dt))

    def bytes_per_random_step(self):
        return int(self._lib.mtfjsp_bytes_per_random_step(self._h, self._dt))

    @property
    def random_step_is_fused(self):
        """True if random_step is one launch (policy + candidate-machine features + step + observation)."""
        return bool(self._lib.mtfjsp_random_step_is_fused(self._h))
