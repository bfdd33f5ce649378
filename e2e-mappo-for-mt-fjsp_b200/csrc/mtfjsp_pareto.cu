// mtfjsp_pareto.cu -- multi-objective kernels for sm_100a over the three targets (mk, ec, tt) of finished schedules:
// a per-segment non-dominated filter, the exact per-segment hypervolume and the per-segment non-dominated sorting rank
// (pareto.py wraps all three).
//
// All three are handle-free and run on the caller's stream.  Points are FP64 [P,3] row-major; segment s is the CSR range
// [seg[s], seg[s+1]).  The filter and the rank are pure comparisons, so their results are exact.  The hypervolume
// restates, operation for operation, the slice sweep documented in include/mtfjsp.h (pareto.hypervolume3_reference is
// the numpy form); this file is built with -fmad=false so that no product is contracted into the sum that follows it.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mtfjsp_launch.cuh"

namespace {

constexpr int FILTER_THREADS = 256;         // candidates per block: one per thread
constexpr int FILTER_WARPS = FILTER_THREADS / 32;
constexpr int FILTER_TILE = 64;             // comparison points per warp tile (two per lane)
constexpr int HV_THREADS = 1024;
constexpr int HV_MAX = 4096;                // points per segment the hypervolume handles (shared-memory bound)
// ux, uy, uz [HV_MAX] f64; term [HV_MAX] f64; zrank, by_z, by_x [HV_MAX] int16; participant flag [HV_MAX] uint8
constexpr size_t HV_SMEM = (size_t)HV_MAX * (4 * sizeof(double) + 3 * sizeof(int16_t) + 1);

__device__ __forceinline__ bool finite3(double a, double b, double c) {
    return isfinite(a) && isfinite(b) && isfinite(c);
}

// grid (S, candidate tiles); block b of segment s takes candidate tiles b, b + gridDim.y, ... of the segment.  Every warp
// streams the segment's points through its own shared tile (no block barrier), and leaves a candidate tile as soon as
// every lane's candidate is settled.
__global__ void __launch_bounds__(FILTER_THREADS) pareto_filter_kernel(const double* __restrict__ obj3,
                                                                      const int64_t* __restrict__ seg,
                                                                      uint8_t* __restrict__ keep) {
    __shared__ double tile[FILTER_WARPS][3][FILTER_TILE];
    const int s = blockIdx.x;
    const int64_t b0 = seg[s], b1 = seg[s + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double (*tw)[FILTER_TILE] = tile[warp];
    for (int64_t c0 = b0 + (int64_t)blockIdx.y * FILTER_THREADS; c0 < b1; c0 += (int64_t)gridDim.y * FILTER_THREADS) {
        const int64_t p = c0 + threadIdx.x;
        const bool mine = p < b1;
        double p0 = 0.0, p1 = 0.0, p2 = 0.0;
        if (mine) {
            p0 = obj3[3 * p]; p1 = obj3[3 * p + 1]; p2 = obj3[3 * p + 2];
        }
        // settled: out of range, non-finite, or dominated / preceded by an equal point
        bool dom = !mine || !finite3(p0, p1, p2);
        if (__all_sync(0xffffffffu, dom)) {
            if (mine) keep[p] = 0;
            continue;
        }
        for (int64_t q0 = b0; q0 < b1; q0 += FILTER_TILE) {
            __syncwarp();
            for (int k = lane; k < FILTER_TILE; k += 32) {
                const int64_t q = q0 + k;
                double v0 = INFINITY, v1 = INFINITY, v2 = INFINITY;  // past the end or non-finite: dominates nothing
                if (q < b1) {
                    v0 = obj3[3 * q]; v1 = obj3[3 * q + 1]; v2 = obj3[3 * q + 2];
                    if (!finite3(v0, v1, v2)) v0 = v1 = v2 = INFINITY;
                }
                tw[0][k] = v0; tw[1][k] = v1; tw[2][k] = v2;
            }
            __syncwarp();
            if (!dom) {
                const int n = (int)(b1 - q0 < FILTER_TILE ? b1 - q0 : FILTER_TILE);
                for (int k = 0; k < n; ++k) {
                    const double v0 = tw[0][k], v1 = tw[1][k], v2 = tw[2][k];
                    const bool le = v0 <= p0 && v1 <= p1 && v2 <= p2;
                    const bool eq = v0 == p0 && v1 == p1 && v2 == p2;
                    dom |= le && (!eq || q0 + k < p);
                }
            }
            if (__all_sync(0xffffffffu, dom)) break;
        }
        if (mine) keep[p] = dom ? 0 : 1;
    }
}

// one block per segment: thread r owns slice r (the participants of z-rank <= r) and sweeps them in x order
__global__ void __launch_bounds__(HV_THREADS) hypervolume3_kernel(const double* __restrict__ obj3,
                                                                 const int64_t* __restrict__ seg,
                                                                 const double* __restrict__ ref3,
                                                                 double* __restrict__ hv) {
    extern __shared__ double smem[];
    double* ux = smem;
    double* uy = ux + HV_MAX;
    double* uz = uy + HV_MAX;
    double* term = uz + HV_MAX;
    int16_t* zrank = reinterpret_cast<int16_t*>(term + HV_MAX);
    int16_t* by_z = zrank + HV_MAX;
    int16_t* by_x = by_z + HV_MAX;
    uint8_t* part = reinterpret_cast<uint8_t*>(by_x + HV_MAX);
    const int s = blockIdx.x;
    const int64_t b0 = seg[s], len = seg[s + 1] - b0;
    const double r0 = ref3[3 * s], r1 = ref3[3 * s + 1], r2 = ref3[3 * s + 2];
    const bool ref_ok = isfinite(r0) && isfinite(r1) && isfinite(r2) && r0 > 0.0 && r1 > 0.0 && r2 > 0.0;
    if (len < 0 || len > HV_MAX || !ref_ok) {
        if (threadIdx.x == 0) hv[s] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const int n = (int)len;
    int count = 0;
    for (int i0 = 0; i0 < n; i0 += HV_THREADS) {
        const int i = i0 + threadIdx.x;
        bool in = false;
        if (i < n) {
            const double a = obj3[3 * (b0 + i)] / r0, b = obj3[3 * (b0 + i) + 1] / r1, c = obj3[3 * (b0 + i) + 2] / r2;
            in = finite3(a, b, c) && a < 1.0 && b < 1.0 && c < 1.0;
            ux[i] = a; uy[i] = b; uz[i] = c;
            part[i] = in;
        }
        count += __syncthreads_count(in);
    }
    // ranks by counting: z by (u_z, index), x by (u_x, u_y, index)
    for (int i = threadIdx.x; i < n; i += HV_THREADS) {
        if (!part[i]) continue;
        const double xi = ux[i], yi = uy[i], zi = uz[i];
        int zr = 0, xr = 0;
        for (int j = 0; j < n; ++j) {
            if (!part[j]) continue;
            const double xj = ux[j], yj = uy[j], zj = uz[j];
            zr += zj < zi || (zj == zi && j < i);
            xr += xj < xi || (xj == xi && (yj < yi || (yj == yi && j < i)));
        }
        zrank[i] = (int16_t)zr;
        by_z[zr] = (int16_t)i;
        by_x[xr] = (int16_t)i;
    }
    __syncthreads();
    for (int r = threadIdx.x; r < count; r += HV_THREADS) {
        double sum = 0.0, m = 1.0, x_prev = 0.0;
        bool any = false;
        for (int k = 0; k < count; ++k) {
            const int j = by_x[k];
            if (zrank[j] > r) continue;
            if (any) sum = sum + (ux[j] - x_prev) * (1.0 - m);
            const double y = uy[j];
            m = y < m ? y : m;
            x_prev = ux[j];
            any = true;
        }
        sum = sum + (1.0 - x_prev) * (1.0 - m);  // slice r holds at least its own point
        const double z_next = r + 1 < count ? uz[by_z[r + 1]] : 1.0;
        term[r] = sum * (z_next - uz[by_z[r]]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        for (int r = 0; r < count; ++r) v = v + term[r];
        hv[s] = v;
    }
}

// Non-dominated sorting, one block per segment (Deb's domination counts): cnt[p] = how many points beat p, one O(n^2)
// pass; then front f + 1 is every point whose count reaches 0 once the beats of front f's members are subtracted, so the
// peeling does O(n^2) work in all.  Shared: the point coordinates when the segment fits `cap` (non-finite rows as NaN,
// which beat nothing), cnt[RANK_MAX] int32 (-1 once ranked), two front lists of RANK_MAX int16 and two list lengths.
constexpr int RANK_THREADS = 1024;
constexpr int RANK_MAX = 4096;              // = HV_MAX: pareto.HV_MAX_POINTS
constexpr size_t RANK_FIXED_SMEM = (size_t)RANK_MAX * (sizeof(int32_t) + 2 * sizeof(int16_t)) + 4 * sizeof(int32_t);

// q beats p: both finite (a NaN coordinate fails every test), q <= p in every coordinate, and q != p or q has the lower
// index -- the filter's relation
__device__ __forceinline__ bool beats(double qx, double qy, double qz, int q, double px, double py, double pz, int p) {
    const bool le = qx <= px && qy <= py && qz <= pz;
    const bool eq = qx == px && qy == py && qz == pz;
    return le && (!eq || q < p);
}

template <bool STAGED>
__device__ void rank_segment(const double* __restrict__ pts, int n, int cap, double* smem, int32_t* __restrict__ rank) {
    double* sx = smem;
    double* sy = sx + cap;
    double* sz = sy + cap;
    int32_t* cnt = reinterpret_cast<int32_t*>(sz + cap);
    int16_t* lists = reinterpret_cast<int16_t*>(cnt + RANK_MAX);  // front list i at lists + i * RANK_MAX
    int32_t* len = reinterpret_cast<int32_t*>(lists + 2 * RANK_MAX);
    auto get = [&](int i, double& x, double& y, double& z) {
        if (STAGED) {
            x = sx[i]; y = sy[i]; z = sz[i];
        } else {
            x = pts[3 * i]; y = pts[3 * i + 1]; z = pts[3 * i + 2];
            if (!finite3(x, y, z)) x = y = z = __longlong_as_double(0x7ff8000000000000LL);
        }
    };
    if (STAGED) {
        for (int i = threadIdx.x; i < n; i += RANK_THREADS) {
            double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
            if (!finite3(x, y, z)) x = y = z = __longlong_as_double(0x7ff8000000000000LL);
            sx[i] = x; sy[i] = y; sz[i] = z;
        }
    }
    if (threadIdx.x == 0) len[0] = len[1] = 0;
    __syncthreads();
    // domination counts; front 0 straight away
    for (int p = threadIdx.x; p < n; p += RANK_THREADS) {
        double px, py, pz;
        get(p, px, py, pz);
        if (isnan(px)) {
            rank[p] = INT32_MAX;
            cnt[p] = -1;
            continue;
        }
        int c = 0;
        for (int q = 0; q < n; ++q) {
            double qx, qy, qz;
            get(q, qx, qy, qz);
            c += beats(qx, qy, qz, q, px, py, pz, p);
        }
        cnt[p] = c;
        if (c == 0) {
            lists[atomicAdd(&len[0], 1)] = (int16_t)p;
            rank[p] = 0;
            cnt[p] = -1;
        }
    }
    __syncthreads();
    int L = len[0];
    for (int f = 0; L > 0; ++f) {
        const int cur = f & 1;
        const int16_t* fr = lists + cur * RANK_MAX;
        // thread p owns cnt[p] for the whole peel
        for (int p = threadIdx.x; p < n; p += RANK_THREADS) {
            if (cnt[p] <= 0) continue;
            double px, py, pz;
            get(p, px, py, pz);
            int d = 0;
            for (int k = 0; k < L; ++k) {
                const int q = fr[k];
                double qx, qy, qz;
                get(q, qx, qy, qz);
                d += beats(qx, qy, qz, q, px, py, pz, p);
            }
            if (d == 0) continue;
            if (cnt[p] == d) {
                lists[(cur ^ 1) * RANK_MAX + atomicAdd(&len[cur ^ 1], 1)] = (int16_t)p;
                rank[p] = f + 1;
                cnt[p] = -1;
            } else {
                cnt[p] -= d;
            }
        }
        // Every thread read this round's L = len[cur] before starting the round, so before this barrier; the barrier
        // also ends the appends to len[cur ^ 1].  After it, len[cur] may be cleared for the next round's appends, and
        // the second barrier orders the clear before them and every read of len[cur ^ 1] before the next round's clear.
        __syncthreads();
        if (threadIdx.x == 0) len[cur] = 0;
        L = len[cur ^ 1];
        __syncthreads();
    }
}

// grid S; segment s ranked in shared memory when it has at most `cap` points, else read from global memory
__global__ void __launch_bounds__(RANK_THREADS) pareto_rank_kernel(const double* __restrict__ obj3,
                                                                  const int64_t* __restrict__ seg, int cap,
                                                                  int32_t* __restrict__ rank) {
    extern __shared__ double rsmem[];
    const int s = blockIdx.x;
    const int64_t b0 = seg[s], len = seg[s + 1] - b0;
    if (len <= 0) return;
    if (len > RANK_MAX) {
        for (int64_t i = threadIdx.x; i < len; i += RANK_THREADS) rank[b0 + i] = -2;
        return;
    }
    if (len <= cap) rank_segment<true>(obj3 + 3 * b0, (int)len, cap, rsmem, rank + b0);
    else rank_segment<false>(obj3 + 3 * b0, (int)len, cap, rsmem, rank + b0);
}

}  // namespace

extern "C" {

int mtfjsp_pareto_filter(const double* obj3, const int64_t* seg, int S, int64_t max_len, uint8_t* keep, void* stream) {
    if (!obj3 || !seg || !keep || S < 0 || max_len < 0) return fail(MTFJSP_E_ARG, "mtfjsp_pareto_filter: bad argument");
    if (S == 0) return MTFJSP_OK;
    const int64_t tiles = (max_len + FILTER_THREADS - 1) / FILTER_THREADS;
    const dim3 grid((unsigned)S, (unsigned)(tiles < 1 ? 1 : (tiles > 65535 ? 65535 : tiles)));
    pareto_filter_kernel<<<grid, FILTER_THREADS, 0, (cudaStream_t)stream>>>(obj3, seg, keep);
    return launched(__func__);
}

int mtfjsp_hypervolume3(const double* obj3, const int64_t* seg, int S, const double* ref3, double* hv, void* stream) {
    if (!obj3 || !seg || !ref3 || !hv || S < 0) return fail(MTFJSP_E_ARG, "mtfjsp_hypervolume3: bad argument");
    if (S == 0) return MTFJSP_OK;
    CK(opt_in_smem(hypervolume3_kernel, HV_SMEM), __func__);
    hypervolume3_kernel<<<(unsigned)S, HV_THREADS, HV_SMEM, (cudaStream_t)stream>>>(obj3, seg, ref3, hv);
    return launched(__func__);
}

int mtfjsp_pareto_rank(const double* obj3, const int64_t* seg, int S, int64_t max_len, int32_t* rank, void* stream) {
    if (!obj3 || !seg || !rank || S < 0 || max_len < 0) return fail(MTFJSP_E_ARG, "mtfjsp_pareto_rank: bad argument");
    if (S == 0) return MTFJSP_OK;
    // coordinates staged for segments up to max_len points (at least one, at most RANK_MAX); longer ones read global
    const int cap = (int)(max_len < 1 ? 1 : (max_len > RANK_MAX ? RANK_MAX : max_len));
    const size_t smem = (size_t)cap * 3 * sizeof(double) + RANK_FIXED_SMEM;
    CK(opt_in_smem(pareto_rank_kernel, smem), __func__);
    pareto_rank_kernel<<<(unsigned)S, RANK_THREADS, smem, (cudaStream_t)stream>>>(obj3, seg, cap, rank);
    return launched(__func__);
}

}  // extern "C"
