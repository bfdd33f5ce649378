// mtfjsp_evolve.cu -- variation operators for sm_100a on (op, machine) action sequences (evolve.py wraps them).
//
// mtfjsp_offspring builds child sequences from parent sequences on the job-sequence view: position s of a sequence holds
// job op_s / M, and each op keeps its machine apart.  A child's job sequence is decoded back to ops by numbering the
// occurrences of each job (position s gets op j * M + the number of earlier occurrences of j), so a child is always a
// complete sequence in job order, and its machines come from the parents or from the op's feasible set: no repair.
//
// One warp per child, with the child's job sequence, the fill list of the crossover, both parents' machines by op, the
// kept-job flags and the per-job counters of the decoder in shared memory (int16 jobs, int8 machines).  Every random draw
// is counter-based, a function of (seed, child, draw index) only, so no result depends on the launch shape.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mtfjsp_launch.cuh"

namespace {

constexpr int OFF_WARPS = 4;  // children per block

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
// draw k of child c: 53 bits -> [0, 1) (the construction of the instance generator's u01)
__device__ __forceinline__ double u01(uint64_t seed, uint64_t c, uint64_t k) {
    const uint64_t x = splitmix64(seed ^ splitmix64(c * 0x100000001B3ULL + k * 0x9E3779B97F4A7C15ULL));
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}
// floor(u * n), clamped to n - 1
__device__ __forceinline__ int below(double u, int n) {
    const int k = (int)(u * (double)n);
    return k < n - 1 ? k : n - 1;
}
// the floor(u * F)-th machine m (in machine order) with t_row[m] >= 0, F of them; -1 when F = 0
__device__ __forceinline__ int nth_feasible(const double* __restrict__ t_row, int M, double u) {
    int F = 0;
    for (int m = 0; m < M; ++m) F += t_row[m] >= 0.0;
    if (F == 0) return -1;
    int k = below(u, F);
    for (int m = 0; m < M; ++m) {
        if (t_row[m] >= 0.0 && k-- == 0) return m;
    }
    return -1;
}

__host__ __device__ __forceinline__ size_t up16(size_t b) { return (b + 15) & ~(size_t)15; }
// child, fill [N] int16; cnt [J] int16; m1, m2 [N] int8; kept [J] uint8
__host__ __device__ __forceinline__ size_t warp_bytes(int J, int M) {
    const size_t N = (size_t)J * M;
    return 2 * up16(2 * N) + up16(2 * (size_t)J) + 2 * up16(N) + up16((size_t)J);
}

__global__ void __launch_bounds__(OFF_WARPS * 32) offspring_kernel(const double* __restrict__ t, int S, int J, int M,
                                                                  const int32_t* __restrict__ parents, int P,
                                                                  const int32_t* __restrict__ pair,
                                                                  const int32_t* __restrict__ inst, int C, uint64_t seed,
                                                                  double p_swap, double p_mach,
                                                                  int32_t* __restrict__ children) {
    extern __shared__ __align__(16) unsigned char osmem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t c = (int64_t)blockIdx.x * OFF_WARPS + w;
    if (c >= C) return;  // warp-uniform
    const int N = J * M;
    unsigned char* base = osmem + w * warp_bytes(J, M);
    int16_t* child = reinterpret_cast<int16_t*>(base);
    int16_t* fill = reinterpret_cast<int16_t*>(base + up16(2 * (size_t)N));
    int16_t* cnt = reinterpret_cast<int16_t*>(base + 2 * up16(2 * (size_t)N));
    int8_t* m1 = reinterpret_cast<int8_t*>(base + 2 * up16(2 * (size_t)N) + up16(2 * (size_t)J));
    int8_t* m2 = m1 + up16(N);
    uint8_t* kept = reinterpret_cast<uint8_t*>(m2 + up16(N));
    int32_t* out = children + (size_t)c * N * 2;
    const unsigned lt = (1u << lane) - 1u;

    const int a = pair[2 * c], b = pair[2 * c + 1], s = inst[c];
    bool bad = s < 0 || s >= S || a < -1 || a >= P || (a >= 0 && (b < 0 || b >= P));
    const int32_t* p1 = parents + (size_t)(a < 0 ? 0 : a) * N * 2;
    const int32_t* p2 = parents + (size_t)(b < 0 ? 0 : b) * N * 2;
    if (!bad && a >= 0) {  // parent entries out of range would index shared memory out of bounds
        bool off = false;
        for (int i = lane; i < N; i += 32) {
            off |= p1[2 * i] < 0 || p1[2 * i] >= N || p1[2 * i + 1] < 0 || p1[2 * i + 1] >= M;
            off |= p2[2 * i] < 0 || p2[2 * i] >= N || p2[2 * i + 1] < 0 || p2[2 * i + 1] >= M;
        }
        bad = __any_sync(0xffffffffu, off);
    }
    if (bad) {
        for (int i = lane; i < 2 * N; i += 32) out[i] = -1;
        return;
    }
    const double* ts = t + (size_t)s * N * M;

    if (a < 0) {
        // random individual: draws [0, N) shuffle the FIFO multiset, [N, 2N) pick each op's machine
        for (int i = lane; i < N; i += 32) {
            child[i] = (int16_t)(i / M);
            m1[i] = (int8_t)nth_feasible(ts + (size_t)i * M, M, u01(seed, c, N + i));
        }
        __syncwarp();
        if (lane == 0) {
            for (int i = N - 1; i > 0; --i) {
                const int k = below(u01(seed, c, i), i + 1);
                const int16_t x = child[i];
                child[i] = child[k];
                child[k] = x;
            }
        }
        __syncwarp();
    } else {
        // POX: draws [0, J) pick the kept jobs; parents' machines by op
        for (int j = lane; j < J; j += 32) kept[j] = u01(seed, c, j) < 0.5;
        for (int i = lane; i < N; i += 32) {
            m1[p1[2 * i]] = (int8_t)p1[2 * i + 1];
            m2[p2[2 * i]] = (int8_t)p2[2 * i + 1];
        }
        __syncwarp();
        // parent 2's non-kept jobs in its order
        int run = 0;
        for (int s0 = 0; s0 < N; s0 += 32) {
            const int i = s0 + lane;
            const int j = i < N ? p2[2 * i] / M : 0;
            const bool take = i < N && !kept[j];
            const unsigned bal = __ballot_sync(0xffffffffu, take);
            if (take) fill[run + __popc(bal & lt)] = (int16_t)j;
            run += __popc(bal);
        }
        __syncwarp();
        // parent 1's kept jobs stay where they are; the other positions take the fill list left to right
        run = 0;
        for (int s0 = 0; s0 < N; s0 += 32) {
            const int i = s0 + lane;
            const int j = i < N ? p1[2 * i] / M : 0;
            const bool other = i < N && !kept[j];
            const unsigned bal = __ballot_sync(0xffffffffu, other);
            if (i < N) child[i] = other ? fill[run + __popc(bal & lt)] : (int16_t)j;
            run += __popc(bal);
        }
        // draws [J, J + N): each op's machine from parent 1 (u < 0.5) or 2; [J + N + 3 + 2o, +1]: reassignment of op o
        for (int o = lane; o < N; o += 32) {
            int m = u01(seed, c, J + o) < 0.5 ? m1[o] : m2[o];
            if (u01(seed, c, J + N + 3 + 2 * o) < p_mach) {
                const int r = nth_feasible(ts + (size_t)o * M, M, u01(seed, c, J + N + 4 + 2 * o));
                if (r >= 0) m = r;
            }
            m1[o] = (int8_t)m;
        }
        __syncwarp();
        // draws J + N .. J + N + 2: the swap of two positions of the job sequence
        if (lane == 0 && u01(seed, c, J + N) < p_swap) {
            const int i = below(u01(seed, c, J + N + 1), N), k = below(u01(seed, c, J + N + 2), N);
            const int16_t x = child[i];
            child[i] = child[k];
            child[k] = x;
        }
        __syncwarp();
    }

    // decode: op = j * M + earlier occurrences of j; lanes of one job in a chunk count among themselves
    for (int j = lane; j < J; j += 32) cnt[j] = 0;
    __syncwarp();
    for (int s0 = 0; s0 < N; s0 += 32) {
        const int i = s0 + lane;
        int j = i < N ? child[i] : -1;
        if (j >= J) j = -1;  // only from parents that are not sequences of this size
        const unsigned peers = __match_any_sync(0xffffffffu, j);
        const int r = __popc(peers & lt);
        const int before = j >= 0 ? cnt[j] : 0;
        __syncwarp();
        if (j >= 0 && r == __popc(peers) - 1) cnt[j] = (int16_t)(before + r + 1);
        __syncwarp();
        if (i < N) {
            const int op = j >= 0 ? j * M + before + r : -1;
            const bool ok = op >= 0 && op < N;
            out[2 * i] = ok ? op : -1;
            out[2 * i + 1] = ok ? m1[op] : -1;
        }
    }
}

}  // namespace

extern "C" {

int mtfjsp_offspring(const double* t, int S, int J, int M, const int32_t* parents, int P, const int32_t* pair,
                     const int32_t* inst, int C, uint64_t seed, double p_swap, double p_mach, int32_t* children,
                     void* stream) {
    if (!t || !parents || !pair || !inst || !children || S < 0 || P < 0 || C < 0 || J < 1 || M < 2 || M > 64 ||
        (int64_t)J * M > 4096)
        return fail(MTFJSP_E_ARG, "mtfjsp_offspring: bad argument");
    if (C == 0) return MTFJSP_OK;
    const size_t smem = OFF_WARPS * warp_bytes(J, M);
    CK(opt_in_smem(offspring_kernel, smem), __func__);
    const unsigned grid = (unsigned)(((int64_t)C + OFF_WARPS - 1) / OFF_WARPS);
    offspring_kernel<<<grid, OFF_WARPS * 32, smem, (cudaStream_t)stream>>>(t, S, J, M, parents, P, pair, inst, C, seed,
                                                                           p_swap, p_mach, children);
    return launched(__func__);
}

}  // extern "C"
