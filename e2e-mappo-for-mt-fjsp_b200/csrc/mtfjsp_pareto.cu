// mtfjsp_pareto.cu -- multi-objective kernels for sm_100a over the three targets (mk, ec, tt) of finished schedules:
// a per-segment non-dominated filter and the exact per-segment hypervolume (pareto.py wraps both).
//
// Both are handle-free and run on the caller's stream.  Points are FP64 [P,3] row-major; segment s is the CSR range
// [seg[s], seg[s+1]).  The filter is pure comparisons, so its bits are exact.  The hypervolume restates, operation for
// operation, the slice sweep documented in include/mtfjsp.h (pareto.hypervolume3_reference is the numpy form); this file
// is built with -fmad=false so that no product is contracted into the sum that follows it.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mtfjsp.h"

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

}  // namespace

extern "C" {

int mtfjsp_pareto_filter(const double* obj3, const int64_t* seg, int S, int64_t max_len, uint8_t* keep, void* stream) {
    if (!obj3 || !seg || !keep || S < 0 || max_len < 0) return MTFJSP_E_ARG;
    if (S == 0) return MTFJSP_OK;
    const int64_t tiles = (max_len + FILTER_THREADS - 1) / FILTER_THREADS;
    const dim3 grid((unsigned)S, (unsigned)(tiles < 1 ? 1 : (tiles > 65535 ? 65535 : tiles)));
    pareto_filter_kernel<<<grid, FILTER_THREADS, 0, (cudaStream_t)stream>>>(obj3, seg, keep);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_hypervolume3(const double* obj3, const int64_t* seg, int S, const double* ref3, double* hv, void* stream) {
    if (!obj3 || !seg || !ref3 || !hv || S < 0) return MTFJSP_E_ARG;
    if (S == 0) return MTFJSP_OK;
    if (cudaFuncSetAttribute(hypervolume3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HV_SMEM) != cudaSuccess)
        return MTFJSP_E_CUDA;
    hypervolume3_kernel<<<(unsigned)S, HV_THREADS, HV_SMEM, (cudaStream_t)stream>>>(obj3, seg, ref3, hv);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

}  // extern "C"
