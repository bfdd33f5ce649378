"""Pareto fronts over the three targets of a finished schedule: makespan mk, energy ec = processing + idle, transport
time tt (the three the reward weights (w_mk, w_ec, w_tt) name).

Every method of the package scores a schedule by one weighted sum; this module keeps the cost vectors apart.  A set of
points is given in CSR form: obj [P,3] f64 and seg [S+1] int64 offsets, segment s = one instance's points
obj[seg[s]:seg[s+1]].  The two hot operations are kernels of csrc/mtfjsp_pareto.cu:

  pareto_filter   the non-dominated points of every segment (mtfjsp_pareto_filter): O(P^2) comparisons per segment, the
                  comparison points streamed through shared memory; of equal points the first is kept;
  hypervolume     the exact hypervolume of every segment inside a per-segment reference point (mtfjsp_hypervolume3), a
                  z-slice sweep of one block per segment, up to 4,096 points.

`pareto_filter_reference` and `hypervolume3_reference` restate both in numpy, expression for expression and in the same
order; they are the specification the kernels are tested against.  `front` and `hypervolume_table` apply the kernels to
the [K,S,4] cost layouts the validators return; `crowding_truncate` is the NSGA-II crowding-distance cut the Pareto local
search (search.pareto_local_search) uses to bound its archive.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check

HV_MAX_POINTS = 4096


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def objectives(final4):
    """[...,4] (mk, pt, tt, idle) costs, numpy or torch -> [...,3] (mk, pt + idle, tt) of the same kind.  pt + idle is
    formed as validate._objective forms it, so w_mk*o[...,0] + w_ec*o[...,1] + w_tt*o[...,2] has its bits."""
    f = final4
    cols = (f[..., 0], f[..., 1] + f[..., 3], f[..., 2])
    return torch.stack(cols, -1) if torch.is_tensor(f) else np.stack(cols, -1)


def _segments(obj, seg, device=None):
    dev = torch.device(device) if device is not None else (obj.device if torch.is_tensor(obj) else torch.device("cuda"))
    if dev.type != "cuda":
        raise ValueError("the Pareto kernels run on a CUDA device")
    o = torch.as_tensor(obj).to(dev, torch.float64).contiguous()
    sg = torch.as_tensor(seg).to(dev, torch.int64).contiguous()
    if o.dim() != 2 or o.shape[1] != 3 or sg.dim() != 1 or sg.shape[0] < 1:
        raise ValueError("obj must have shape [P, 3] and seg [S + 1]")
    return o, sg


def pareto_filter(obj, seg, max_len=None):
    """Non-dominated points of every segment (mtfjsp_pareto_filter): bool keep [P] on the device.  obj [P,3], seg [S+1]
    (torch or numpy; the device of obj, else cuda).  max_len: the longest segment, if known (else one synchronisation
    reads it); it sizes the grid only."""
    o, sg = _segments(obj, seg)
    S = sg.shape[0] - 1
    if max_len is None:
        max_len = int((sg[1:] - sg[:-1]).max()) if S else 0
    keep = torch.zeros((o.shape[0],), dtype=torch.uint8, device=o.device)
    if o.shape[0] == 0:  # nothing to write (and an empty tensor may have no address)
        return keep.bool()
    check(_lib.lib().mtfjsp_pareto_filter(_ptr(o), _ptr(sg), S, int(max_len), _ptr(keep), _stream()),
          "mtfjsp_pareto_filter")
    return keep.bool()


def hypervolume(obj, seg, ref):
    """Exact hypervolume of every segment inside its reference point (mtfjsp_hypervolume3): [S] f64 on the device, in
    units of the box ref (the points are divided by ref[s]).  obj [P,3], seg [S+1], ref [S,3].  NaN for a segment of more
    than 4,096 points or a ref row that is not finite and > 0."""
    o, sg = _segments(obj, seg)
    S = sg.shape[0] - 1
    r = torch.as_tensor(ref).to(o.device, torch.float64).contiguous()
    if tuple(r.shape) != (S, 3):
        raise ValueError("ref must have shape [%d, 3]" % S)
    hv = torch.empty((S,), dtype=torch.float64, device=o.device)
    if S == 0:
        return hv
    if o.shape[0] == 0:  # every segment empty: a stand-in row gives the kernel an address it never reads
        o = torch.zeros((1, 3), dtype=torch.float64, device=o.device)
    check(_lib.lib().mtfjsp_hypervolume3(_ptr(o), _ptr(sg), S, _ptr(r), _ptr(hv), _stream()), "mtfjsp_hypervolume3")
    return hv


def _layout(final4):
    f = torch.as_tensor(np.asarray(final4) if not torch.is_tensor(final4) else final4, dtype=torch.float64)
    if f.dim() == 2:
        f = f[None]
    if f.dim() != 3 or f.shape[2] != 4:
        raise ValueError("final4 must have shape [S, 4] or [K, S, 4]")
    return f


def front(final4, device=None):
    """The per-instance Pareto front of [K,S,4] costs (the final4 layout of sampled_validate and beam_validate; [S,4]
    is K = 1): a list of S int64 numpy arrays of indices into K, ascending (of equal cost vectors the lowest k)."""
    f = _layout(final4)
    K, S = f.shape[0], f.shape[1]
    o = objectives(f.transpose(0, 1).reshape(S * K, 4))
    seg = torch.arange(S + 1, dtype=torch.int64) * K
    keep = pareto_filter(o.to(device or "cuda"), seg, K).cpu().numpy().reshape(S, K)
    return [np.nonzero(keep[s])[0] for s in range(S)]


def reference_point(obj):
    """1.1 x the componentwise max of the finite points of obj [..., S, 3] over its leading axes -> [S,3]; 1.0 where
    that max is 0 or there is no finite point."""
    o = np.asarray(obj, dtype=np.float64).reshape(-1, *np.shape(obj)[-2:])
    mx = np.where(np.isfinite(o).all(-1, keepdims=True), o, -np.inf).max(axis=0)
    return np.where((mx == 0) | (mx == -np.inf), 1.0, 1.1 * mx)


def hypervolume_table(sets, device=None):
    """Hypervolume of each method's schedules per instance, in one shared per-instance reference point.
    sets: {method name: final4 [S,4] or [K,S,4]} over the same S instances.  The reference point of an instance is
    1.1 x the componentwise max of (mk, ec, tt) over the union of all methods' points, 1.0 where that max is 0.
    -> dict: hypervolume {name: [S]}, union [S] (the hypervolume of all methods' points together), ref [S,3], numpy."""
    objs = {k: objectives(_layout(v)).numpy() for k, v in sets.items()}     # [K,S,3] each
    S = next(iter(objs.values())).shape[1]
    if any(o.shape[1] != S for o in objs.values()):
        raise ValueError("every method must cover the same instances")
    allp = np.concatenate(list(objs.values()), axis=0)                       # [sum K, S, 3]
    ref = reference_point(allp)
    dev = device or "cuda"

    def hv(o):  # [K,S,3] -> [S]; the front first, so any number of points fits the kernel's 4,096
        K = o.shape[0]
        pts = torch.as_tensor(o.transpose(1, 0, 2).reshape(S * K, 3), device=dev)
        seg = torch.arange(S + 1, dtype=torch.int64, device=dev) * K
        keep = pareto_filter(pts, seg, K)
        cnt = keep.view(S, K).sum(1)
        seg2 = torch.cat((torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(cnt, 0)))
        return hypervolume(pts[keep], seg2, ref).cpu().numpy()

    return {"hypervolume": {k: hv(o) for k, o in objs.items()}, "union": hv(allp), "ref": ref}


def crowding_distance(obj, inst, S):
    """NSGA-II crowding distance of every point of obj [P,3] (torch, any device) within its group inst [P] int64 (groups
    0 .. S-1, any order) -> [P] f64.  Per objective in the order mk, ec, tt: the group's points sorted ascending (ties:
    lower index first); the first and last get +inf, an interior point adds (v_next - v_prev) / (v_max - v_min), or 0
    where v_max == v_min, to a sum from 0.0."""
    P = obj.shape[0]
    dev = obj.device
    cd = torch.zeros((P,), dtype=torch.float64, device=dev)
    if P == 0:
        return cd
    for d in range(3):
        v = obj[:, d]
        o = torch.sort(v, stable=True)[1]
        o = o[torch.sort(inst[o], stable=True)[1]]                           # by (group, value, index)
        g, vs = inst[o], v[o]
        first = torch.ones((P,), dtype=torch.bool, device=dev)
        last = torch.ones((P,), dtype=torch.bool, device=dev)
        first[1:] = g[1:] != g[:-1]
        last[:-1] = g[:-1] != g[1:]
        vmin = torch.full((S,), float("inf"), dtype=torch.float64, device=dev).scatter_reduce(0, g, vs, "amin")
        vmax = torch.full((S,), float("-inf"), dtype=torch.float64, device=dev).scatter_reduce(0, g, vs, "amax")
        span = (vmax - vmin)[g]
        nxt = torch.cat((vs[1:], vs[-1:]))
        prv = torch.cat((vs[:1], vs[:-1]))
        inner = torch.where(span == 0, torch.zeros_like(vs), (nxt - prv) / torch.where(span == 0, 1.0, span))
        term = torch.where(first | last, float("inf"), inner)
        cd[o] = cd[o] + term
    return cd


def crowding_truncate(obj, inst, S, cap):
    """The points crowding_truncate keeps: bool [P].  In every group of more than `cap` points, the `cap` points of the
    largest crowding distance (ties: the lower index); every point of a smaller group."""
    P = obj.shape[0]
    if P == 0:
        return torch.zeros((0,), dtype=torch.bool, device=obj.device)
    cd = crowding_distance(obj, inst, S)
    o = torch.sort(cd, descending=True, stable=True)[1]
    o = o[torch.sort(inst[o], stable=True)[1]]
    cnt = torch.bincount(inst, minlength=S)
    start = torch.cumsum(cnt, 0) - cnt
    rank = torch.empty_like(o)
    rank[o] = torch.arange(P, device=obj.device) - start[inst[o]]
    return rank < cap


# --------------------------------------------------------------------------------------- numpy specification (reference)
def pareto_filter_reference(obj, seg):
    """numpy restatement of mtfjsp_pareto_filter: keep [P] bool, the kernel's comparisons."""
    obj = np.asarray(obj, dtype=np.float64)
    seg = np.asarray(seg, dtype=np.int64)
    keep = np.zeros(obj.shape[0], dtype=bool)
    for s in range(len(seg) - 1):
        a, b = int(seg[s]), int(seg[s + 1])
        if b <= a:
            continue
        p = obj[a:b]
        fin = np.isfinite(p).all(axis=1)
        q = np.where(fin[:, None], p, np.inf)                               # non-finite: dominates nothing
        idx = np.arange(b - a)
        dom = ~fin
        for c0 in range(0, b - a, 512):                                     # candidates c0 .. c0+511 against all q
            pc = p[c0:c0 + 512]
            le = (q[None, :, :] <= pc[:, None, :]).all(-1)
            eq = (q[None, :, :] == pc[:, None, :]).all(-1)
            dom[c0:c0 + 512] |= (le & (~eq | (idx[None, :] < idx[c0:c0 + 512, None]))).any(1)
        keep[a:b] = ~dom
    return keep


def hypervolume3_reference(obj, seg, ref):
    """numpy restatement of mtfjsp_hypervolume3, operation for operation and in the kernel's order: [S] f64."""
    obj = np.asarray(obj, dtype=np.float64)
    seg = np.asarray(seg, dtype=np.int64)
    ref = np.asarray(ref, dtype=np.float64)
    S = len(seg) - 1
    hv = np.zeros(S)
    for s in range(S):
        a, b = int(seg[s]), int(seg[s + 1])
        r = ref[s]
        if b - a < 0 or b - a > HV_MAX_POINTS or not (np.isfinite(r).all() and (r > 0).all()):
            hv[s] = np.nan
            continue
        u = obj[a:b] / r
        u = u[np.isfinite(u).all(axis=1) & (u < 1.0).all(axis=1)]          # participants, in index order
        n = len(u)
        if n == 0:
            continue
        idx = np.arange(n)
        by_z = np.lexsort((idx, u[:, 2]))
        zrank = np.empty(n, dtype=np.int64)
        zrank[by_z] = idx
        by_x = np.lexsort((idx, u[:, 1], u[:, 0]))
        zr_x = zrank[by_x]
        z = np.append(u[by_z, 2], 1.0)
        total = 0.0
        for i in range(n):
            pts = by_x[zr_x <= i]
            xs = u[pts, 0]
            m = np.minimum.accumulate(u[pts, 1])                            # min(1.0, u_y) = u_y for a participant
            xn = np.append(xs[1:], 1.0)
            area = np.add.accumulate((xn - xs) * (1.0 - m))[-1]             # sequential, from the first term
            total = total + area * (z[i + 1] - z[i])
        hv[s] = total
    return hv
