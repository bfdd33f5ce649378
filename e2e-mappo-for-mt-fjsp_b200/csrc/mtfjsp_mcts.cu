// mtfjsp_mcts.cu -- Monte Carlo tree search over joint (op, machine) actions for sm_100a (search.mcts_search wraps it).
//
// S trees, one per instance, each a pool of P nodes in caller-owned device arrays.  A node holds NODE_FIELDS int32
// (parent, first child, child count, edge op, edge machine, visits, virtual visits) and one f64 vmin, the least objective
// backed up through it.  Children of a node are one contiguous block in flat candidate order, allocated when the node is
// expanded.  No env state is stored: a node is the path of actions from the root, and its leaf is scored by
// mtfjsp_complete with that path as forced actions.
//
// mtfjsp_mcts_select runs one warp per tree and makes the L selections of a round in order; the candidates of a node are
// derived from the root's next op of every job plus the path's actions, one lane per job (the per-job counters in
// shared memory).  mtfjsp_mcts_backup runs one thread per tree and walks the L paths serially.  Built with -fmad=false:
// the score is restated in numpy (search.mcts_reference) bit for bit.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "mtfjsp_launch.cuh"

namespace {

constexpr int SEL_WARPS = 4;      // trees per block of the selection
constexpr int BACKUP_THREADS = 128;
constexpr unsigned FULL = 0xffffffffu;
enum { PARENT = 0, FIRST = 1, NCHILD = 2, OP = 3, MACH = 4, VISITS = 5, VIRTUAL = 6, F = 7 };

// feasible children of job j at its next op k (0 <= k < M, else none): every machine with t >= 0 ("all", rule == NULL),
// or the rule table's machine when t >= 0 there
__device__ __forceinline__ int job_children(const double* __restrict__ ts, const int32_t* __restrict__ rule, int j, int k,
                                            int M) {
    if (k < 0 || k >= M) return 0;
    const int op = j * M + k;
    const double* tr = ts + (size_t)op * M;
    if (rule) {
        const int m = rule[op];
        return m >= 0 && m < M && tr[m] >= 0.0;
    }
    int n = 0;
#pragma unroll 1
    for (int m = 0; m < M; ++m) n += tr[m] >= 0.0;
    return n;
}

// inclusive warp scan of x
__device__ __forceinline__ int warp_scan(int x, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(FULL, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

__global__ void __launch_bounds__(SEL_WARPS * 32) mcts_select_kernel(
    const double* __restrict__ t, const int32_t* __restrict__ rule, int S, int J, int M, const int32_t* __restrict__ next0,
    int L, int P, int D, double c, int32_t* __restrict__ node, double* __restrict__ vmin, const int32_t* __restrict__ root,
    int32_t* __restrict__ count, const double* __restrict__ lohi, int32_t* __restrict__ paths, int32_t* __restrict__ depth,
    int32_t* __restrict__ leaf) {
    extern __shared__ int32_t sel_nx[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x * SEL_WARPS + w;
    if (s >= S) return;  // warp-uniform
    const int N = J * M;
    int32_t* nx = sel_nx + (size_t)w * J;
    int32_t* nd = node + (size_t)s * P * F;
    double* vm = vmin + (size_t)s * P;
    const double* ts = t + (size_t)s * N * M;
    const int32_t* rs = rule ? rule + (size_t)s * N : nullptr;
    const double lo = lohi[2 * s], hi = lohi[2 * s + 1];
    int cnt = count[s];
    const int r0 = root[s];
    const bool tree_ok = cnt >= 1 && cnt <= P && r0 >= 0 && r0 < cnt;

    for (int l = 0; l < L; ++l) {
        const size_t row = (size_t)s * L + l;
        int32_t* pa = paths + row * D * 2;
        for (int j = lane; j < J; j += 32) nx[j] = next0[(size_t)s * J + j];
        __syncwarp();
        int x = tree_ok ? r0 : -1, d = 0;
        while (x >= 0) {
            const int32_t* xn = nd + (size_t)x * F;
            const int seen = xn[VISITS] + xn[VIRTUAL];
            int fc = xn[FIRST], nc = xn[NCHILD];
            __syncwarp();
            if (lane == 0) nd[(size_t)x * F + VIRTUAL] = xn[VIRTUAL] + 1;
            __syncwarp();
            int child = -1;
            if (fc == -1 && nc == 0) {  // unexpanded: a leaf unless it was reached before and its block fits
                if (seen == 0 || d >= D) break;
                int total = 0;
                for (int j0 = 0; j0 < J; j0 += 32) {
                    const int j = j0 + lane;
                    const int n = j < J ? job_children(ts, rs, j, nx[j], M) : 0;
                    total += __reduce_add_sync(FULL, (unsigned)n);
                }
                if (total == 0 || total > P - cnt) break;  // terminal, or the pool is full
                int base = cnt;
                for (int j0 = 0; j0 < J; j0 += 32) {
                    const int j = j0 + lane;
                    const int k = j < J ? nx[j] : -1;
                    const int n = j < J ? job_children(ts, rs, j, k, M) : 0;
                    const int incl = warp_scan(n, lane);
                    if (n > 0) {
                        int at = base + incl - n;
                        const int op = j * M + k;
#pragma unroll 1
                        for (int m = 0; m < M; ++m) {
                            const bool take = rs ? m == rs[op] : ts[(size_t)op * M + m] >= 0.0;
                            if (!take) continue;
                            int32_t* cn = nd + (size_t)at * F;
                            cn[PARENT] = x; cn[FIRST] = -1; cn[NCHILD] = 0; cn[OP] = op; cn[MACH] = m;
                            cn[VISITS] = 0; cn[VIRTUAL] = 0;
                            vm[at] = INFINITY;
                            ++at;
                        }
                    }
                    base += __shfl_sync(FULL, incl, 31);
                }
                if (lane == 0) {
                    nd[(size_t)x * F + FIRST] = cnt;
                    nd[(size_t)x * F + NCHILD] = total;
                }
                child = cnt;
                cnt += total;
                __syncwarp();
            } else {
                if (fc < 0 || nc < 1 || fc > cnt - nc || d >= D) break;  // a malformed block is data: a leaf
                // the lowest child nothing has reached, else the largest score, ties to the lowest
                const double u = c * sqrt((double)(seen + 1));
                int fresh = nc;
                double best = -INFINITY;
                int bi = nc;
                for (int i = lane; i < nc; i += 32) {
                    const int32_t* cn = nd + (size_t)(fc + i) * F;
                    const int n = cn[VISITS], v = cn[VIRTUAL];
                    if (n + v == 0) {
                        fresh = min(fresh, i);
                        continue;
                    }
                    const double vc = vm[fc + i];
                    const double q = vc == INFINITY ? 0.0 : (hi == lo ? 1.0 : (hi - vc) / (hi - lo));
                    const double sc = q * (double)n / (double)(n + v) + u / (double)(1 + n + v);
                    if (sc > best || bi == nc) {
                        best = sc;
                        bi = i;
                    }
                }
                fresh = __reduce_min_sync(FULL, (unsigned)fresh);
                if (fresh < nc) {
                    child = fc + fresh;
                } else {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const double b2 = __shfl_xor_sync(FULL, best, o);
                        const int i2 = __shfl_xor_sync(FULL, bi, o);
                        if (i2 < nc && (bi == nc || b2 > best || (b2 == best && i2 < bi))) {
                            best = b2;
                            bi = i2;
                        }
                    }
                    child = fc + bi;
                }
            }
            // step into the child: its edge action extends the path and advances its job
            const int op = nd[(size_t)child * F + OP], m = nd[(size_t)child * F + MACH];
            if (lane == 0) {
                pa[2 * d] = op;
                pa[2 * d + 1] = m;
                if (op >= 0 && op < N) nx[op / M] += 1;
            }
            __syncwarp();
            ++d;
            x = child;
        }
        for (int i = 2 * d + lane; i < 2 * D; i += 32) pa[i] = -1;
        if (lane == 0) {
            depth[row] = d;
            leaf[row] = x;
        }
        __syncwarp();
    }
    if (lane == 0) count[s] = cnt;
}

__global__ void __launch_bounds__(BACKUP_THREADS) mcts_backup_kernel(int S, int L, int P, const int32_t* __restrict__ leaf,
                                                                   const double* __restrict__ obj, int32_t* __restrict__ node,
                                                                   double* __restrict__ vmin, const int32_t* __restrict__ root,
                                                                   const int32_t* __restrict__ count,
                                                                   double* __restrict__ lohi) {
    const int s = blockIdx.x * BACKUP_THREADS + threadIdx.x;
    if (s >= S) return;
    int32_t* nd = node + (size_t)s * P * F;
    double* vm = vmin + (size_t)s * P;
    const int r0 = root[s], cnt = min(count[s], P);
    double lo = lohi[2 * s], hi = lohi[2 * s + 1];
    for (int l = 0; l < L; ++l) {
        const size_t row = (size_t)s * L + l;
        const double v = obj[row];
        int x = leaf[row];
        if (x < 0 || x >= cnt) continue;
        for (int k = 0; k < cnt; ++k) {  // at most cnt nodes on a path: a cycle in malformed data ends here
            int32_t* xn = nd + (size_t)x * F;
            xn[VISITS] += 1;
            xn[VIRTUAL] -= 1;
            if (v < vm[x]) vm[x] = v;
            if (x == r0) break;
            x = xn[PARENT];
            if (x < 0 || x >= cnt) break;
        }
        if (isfinite(v)) {
            lo = v < lo ? v : lo;
            hi = v > hi ? v : hi;
        }
    }
    lohi[2 * s] = lo;
    lohi[2 * s + 1] = hi;
}

}  // namespace

extern "C" {

int mtfjsp_mcts_select(const double* t, const int32_t* rule_mach, int S, int J, int M, const int32_t* next_op, int L,
                       int max_nodes, int max_depth, double c, int32_t* node, double* vmin, const int32_t* root,
                       int32_t* count, const double* lohi, int32_t* paths, int32_t* depth, int32_t* leaf, void* stream) {
    if (!t || !next_op || !node || !vmin || !root || !count || !lohi || !paths || !depth || !leaf || S < 1 || L < 1 ||
        max_nodes < 1 || max_depth < 0 || J < 1 || M < 2 || M > 64 || (int64_t)J * M > 4096)
        return fail(MTFJSP_E_ARG, "mtfjsp_mcts_select: bad argument");
    const size_t smem = (size_t)SEL_WARPS * J * sizeof(int32_t);
    CK(opt_in_smem(mcts_select_kernel, smem), __func__);
    const unsigned grid = (unsigned)((S + SEL_WARPS - 1) / SEL_WARPS);
    mcts_select_kernel<<<grid, SEL_WARPS * 32, smem, (cudaStream_t)stream>>>(t, rule_mach, S, J, M, next_op, L, max_nodes,
                                                                            max_depth, c, node, vmin, root, count, lohi,
                                                                            paths, depth, leaf);
    return launched(__func__);
}

int mtfjsp_mcts_backup(int S, int L, int max_nodes, const int32_t* leaf, const double* objective, int32_t* node,
                       double* vmin, const int32_t* root, const int32_t* count, double* lohi, void* stream) {
    if (!leaf || !objective || !node || !vmin || !root || !count || !lohi || S < 1 || L < 1 || max_nodes < 1)
        return fail(MTFJSP_E_ARG, "mtfjsp_mcts_backup: bad argument");
    const unsigned grid = (unsigned)((S + BACKUP_THREADS - 1) / BACKUP_THREADS);
    mcts_backup_kernel<<<grid, BACKUP_THREADS, 0, (cudaStream_t)stream>>>(S, L, max_nodes, leaf, objective, node, vmin,
                                                                          root, count, lohi);
    return launched(__func__);
}

}  // extern "C"
