// mtfjsp_tabu.cu -- one tabu-search iteration's move decision for sm_100a (search.tabu_search wraps it).
//
// S instances, each with a current schedule, the best schedule seen, and a tabu memory in caller-owned device arrays.
// One warp per instance (one warp per block) stages the current sequence in shared memory, scans the instance's segment
// of the iteration's moves for the admissible move of the least objective, and applies it in place: the new sequence is
// written from the staged copy, so no entry is read after it was overwritten.  Everything is integer work and copies of
// the caller's doubles; search.tabu_reference restates it in numpy exactly.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mtfjsp_launch.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;

struct TabuArgs {
    int S, N, M;
    const int32_t* moves;
    int64_t R;
    const int64_t* seg;
    const double *obj, *f4;
    int it, until_mach, until_ins;  // it + 1 + tenure
    int32_t* cur;
    double *cur_obj, *cur_f4;
    int32_t* best;
    double *best_obj, *best_f4;
    int32_t *mach_until, *op_until, *chosen;
};

__global__ void __launch_bounds__(32) tabu_move_kernel(const __grid_constant__ TabuArgs A) {
    extern __shared__ int32_t tabu_row[];  // [N,2]: the instance's current sequence before the move
    const int s = blockIdx.x, lane = threadIdx.x;
    const int N = A.N, M = A.M;
    int32_t* cs = A.cur + (size_t)s * N * 2;
    for (int i = lane; i < 2 * N; i += 32) tabu_row[i] = cs[i];
    __syncwarp();
    const int64_t lo = A.seg[s], hi = A.seg[s + 1];
    if (lo < 0 || hi < lo || hi > A.R) {  // a malformed segment is data: the instance stays put
        if (lane == 0) A.chosen[s] = -2;
        return;
    }
    const double bo = A.best_obj[s];
    const int32_t* mu = A.mach_until + (size_t)s * N * M;
    const int32_t* ou = A.op_until + (size_t)s * N;
    // per lane the admissible move of the least objective among r = lo + lane + 32k; increasing r keeps the first of
    // equal objectives
    double v = 0.0;
    int64_t bi = -1;
    for (int64_t r = lo + lane; r < hi; r += 32) {
        const int32_t* mv = A.moves + r * 4;
        const int row = mv[0], kind = mv[1], ms = mv[2], arg = mv[3];
        if (row != s || ms < 0 || ms >= N) continue;
        const int o = tabu_row[2 * ms];
        if (o < 0 || o >= N) continue;
        bool tabu;
        if (kind == 0) {
            const int mo = tabu_row[2 * ms + 1];
            if (arg < 0 || arg >= M || mo < 0 || mo >= M) continue;
            tabu = mu[(size_t)o * M + arg] > A.it;
        } else if (kind == 1) {
            if (arg < 0 || arg >= N) continue;
            tabu = ou[o] > A.it;
        } else {
            continue;
        }
        const double x = A.obj[r];
        if (x != x || (tabu && !(x < bo))) continue;  // NaN never wins; a tabu move needs aspiration
        if (bi < 0 || x < v) {
            v = x;
            bi = r;
        }
    }
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) {
        const double v2 = __shfl_xor_sync(FULL, v, k);
        const int64_t b2 = __shfl_xor_sync(FULL, bi, k);
        if (b2 >= 0 && (bi < 0 || v2 < v || (v2 == v && b2 < bi))) {
            v = v2;
            bi = b2;
        }
    }
    if (bi < 0) {  // no admissible move, or an empty segment
        if (lane == 0) A.chosen[s] = -1;
        return;
    }
    const int32_t* mv = A.moves + bi * 4;
    const int kind = mv[1], ms = mv[2], arg = mv[3];
    const bool ins = kind == 1, better = v < bo;
    int32_t* bs = A.best + (size_t)s * N * 2;
    for (int n = lane; n < N; n += 32) {  // search.apply_moves' index arithmetic
        int from = n;
        if (ins) {
            const int rest = n < arg ? n : n - 1;
            from = n == arg ? ms : (rest < ms ? rest : rest + 1);
        }
        const int op = tabu_row[2 * from], m = !ins && n == ms ? arg : tabu_row[2 * from + 1];
        cs[2 * n] = op;
        cs[2 * n + 1] = m;
        if (better) {
            bs[2 * n] = op;
            bs[2 * n + 1] = m;
        }
    }
    if (lane < 4) {
        const double y = A.f4[bi * 4 + lane];
        A.cur_f4[(size_t)s * 4 + lane] = y;
        if (better) A.best_f4[(size_t)s * 4 + lane] = y;
    }
    if (lane == 0) {
        const int o = tabu_row[2 * ms];
        if (ins) A.op_until[(size_t)s * N + o] = A.until_ins;
        else A.mach_until[((size_t)s * N + o) * M + tabu_row[2 * ms + 1]] = A.until_mach;
        A.cur_obj[s] = v;
        if (better) A.best_obj[s] = v;
        A.chosen[s] = (int32_t)bi;
    }
}

}  // namespace

extern "C" {

int mtfjsp_tabu_move(int S, int J, int M, const int32_t* moves, int64_t R, const int64_t* seg, const double* obj,
                     const double* f4, int it, int tenure_mach, int tenure_ins, int32_t* cur, double* cur_obj,
                     double* cur_f4, int32_t* best, double* best_obj, double* best_f4, int32_t* mach_until,
                     int32_t* op_until, int32_t* chosen, void* stream) {
    if (S < 1 || J < 1 || M < 2 || M > 64 || (int64_t)J * M > 4096 || R < 0 || R > INT32_MAX ||
        (R > 0 && (!moves || !obj || !f4)) || !seg || !cur || !cur_obj || !cur_f4 || !best || !best_obj || !best_f4 ||
        !mach_until || !op_until || !chosen || it < 0 || tenure_mach < 0 || tenure_ins < 0 ||
        (int64_t)it + 1 + tenure_mach > INT32_MAX || (int64_t)it + 1 + tenure_ins > INT32_MAX)
        return fail(MTFJSP_E_ARG, "mtfjsp_tabu_move: bad argument");
    TabuArgs A;
    A.S = S; A.N = J * M; A.M = M;
    A.moves = moves; A.R = R; A.seg = seg; A.obj = obj; A.f4 = f4;
    A.it = it; A.until_mach = it + 1 + tenure_mach; A.until_ins = it + 1 + tenure_ins;
    A.cur = cur; A.cur_obj = cur_obj; A.cur_f4 = cur_f4;
    A.best = best; A.best_obj = best_obj; A.best_f4 = best_f4;
    A.mach_until = mach_until; A.op_until = op_until; A.chosen = chosen;
    const size_t smem = (size_t)A.N * 2 * sizeof(int32_t);  // at most 32 KB: no opt-in
    tabu_move_kernel<<<S, 32, smem, (cudaStream_t)stream>>>(A);
    return launched(__func__);
}

}  // extern "C"
