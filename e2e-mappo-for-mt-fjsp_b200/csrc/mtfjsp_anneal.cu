// mtfjsp_anneal.cu -- parallel tempering over finished schedules for sm_100a (search.anneal_search wraps it).
//
// S instances with K Markov chains each; chain row q = s*K + k holds a complete (op, machine) sequence.  Every iteration
// each chain proposes one uniformly drawn neighbour (mtfjsp_anneal_propose), the caller replays it (mtfjsp_replay_moves),
// and mtfjsp_anneal_step takes or rejects it by the Metropolis rule, exchanges adjacent temperatures' states and keeps
// the best state visited.  Every draw is counter-based on (seed, it, k), without the instance row, so an instance's run
// depends neither on the batch nor on its row in it.  The acceptance test uses exp_neg below, built from correctly
// rounded +, -, *, / and exact scaling only, so this file is compiled with -fmad=false and search.exp_neg_reference
// restates it bit for bit in numpy; the rest is integer work and copies of the caller's doubles.
#include <cuda_runtime.h>
#include <stdint.h>

#include "mtfjsp_launch.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int MAX_WARPS = 8;

// evolve._draws' layout: draw j of counter c
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__device__ __forceinline__ double u01(uint64_t seed, uint64_t c, uint64_t j) {
    const uint64_t x = splitmix64(seed ^ splitmix64(c * 0x100000001B3ULL + j * 0x9E3779B97F4A7C15ULL));
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}
// chain k's counter at iteration it
__device__ __forceinline__ uint64_t chain_counter(int it, int k) { return ((uint64_t)(uint32_t)it << 32) | (uint32_t)k; }

// e^-x for x > 0, 1 for x <= 0, NaN for NaN: Cody-Waite reduction x = n ln2 + r, |r| <= ln2/2, the degree-13 Taylor
// polynomial of e^z at z = -r in Horner form, then an exact scaling by 2^-n; 0 past 746
constexpr double INV_LN2 = 1.4426950408889634;
constexpr double LN2_HI = 0.6931471803691238;     // 0x3fe62e42fee00000: n * LN2_HI is exact for n < 2^21
constexpr double LN2_LO = 1.9082149292705877e-10;
constexpr double EXP_NEG_ZERO = 746.0;
__device__ __forceinline__ double exp_neg(double x) {
    if (x != x) return x;
    if (x <= 0.0) return 1.0;
    if (x > EXP_NEG_ZERO) return 0.0;
    const double n = rint(x * INV_LN2);
    const double z = -((x - n * LN2_HI) - n * LN2_LO);
    double p = 1.6059043836821613e-10;  // 1/13!
    p = p * z + 2.08767569878681e-09;
    p = p * z + 2.505210838544172e-08;
    p = p * z + 2.755731922398589e-07;
    p = p * z + 2.7557319223985893e-06;
    p = p * z + 2.48015873015873e-05;
    p = p * z + 0.0001984126984126984;
    p = p * z + 0.001388888888888889;
    p = p * z + 0.008333333333333333;
    p = p * z + 0.041666666666666664;
    p = p * z + 0.16666666666666666;
    p = p * z + 0.5;
    p = p * z + 1.0;
    p = p * z + 1.0;
    return scalbn(p, -(int)n);
}

// floor(u * n), clamped to n - 1
__device__ __forceinline__ int64_t below(double u, int64_t n) {
    const int64_t k = (int64_t)(u * (double)n);
    return k < n - 1 ? k : n - 1;
}

// ---- proposal --------------------------------------------------------------------------------------------------------
// one warp per chain; per warp in shared memory pos [N] (index of op o in the row), and per entry the number of its
// reassignments cre [N] and insertions cin [N]
__host__ __device__ __forceinline__ size_t propose_warp_bytes(int N) { return (size_t)3 * N * sizeof(int32_t); }

struct ProposeArgs {
    const double* t;
    int S, N, M, K, it;
    int64_t Q;  // S * K
    const int32_t* cur;
    uint64_t seed;
    int32_t* moves;
};

// the entry n and offset r of draw `idx` among the per-entry counts c[0..N): sum c[0..n) <= idx < sum c[0..n]
__device__ __forceinline__ void find_entry(const int32_t* c, int N, int64_t idx, int lane, int& n_out, int64_t& r_out) {
    int64_t run = 0;
    for (int b = 0; b < N; b += 32) {
        const int n = b + lane;
        const int64_t x = n < N ? c[n] : 0;
        int64_t inc = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t y = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += y;
        }
        const unsigned hit = __ballot_sync(FULL, run + inc > idx && run + inc - x <= idx && x > 0);
        if (hit) {
            const int src = __ffs(hit) - 1;
            n_out = b + src;
            r_out = idx - run - __shfl_sync(FULL, inc - x, src);
            return;
        }
        run += __shfl_sync(FULL, inc, 31);
    }
    n_out = -1;
    r_out = 0;
}

__global__ void __launch_bounds__(MAX_WARPS * 32) anneal_propose_kernel(const __grid_constant__ ProposeArgs A) {
    extern __shared__ int32_t prop_smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + w;
    if (q >= A.Q) return;  // warp-uniform
    const int N = A.N, M = A.M;
    const int s = (int)(q / A.K), k = (int)(q % A.K);
    int32_t* pos = prop_smem + (size_t)w * 3 * N;
    int32_t* cre = pos + N;
    int32_t* cin = cre + N;
    const int32_t* row = A.cur + (size_t)q * N * 2;
    const double* ts = A.t + (size_t)s * N * M;
    int32_t* out = A.moves + q * 4;

    // the row must be a permutation of the ops: pos of every op, then every entry must own its op's slot
    for (int o = lane; o < N; o += 32) pos[o] = -1;
    __syncwarp();
    bool bad = false;
    for (int n = lane; n < N; n += 32) {
        const int o = row[2 * n];
        if (o < 0 || o >= N) bad = true;
        else pos[o] = n;
    }
    __syncwarp();
    for (int n = lane; n < N && !bad; n += 32) bad = pos[row[2 * n]] != n;
    if (__any_sync(FULL, bad)) {
        if (lane == 0) {
            out[0] = (int32_t)q; out[1] = -1; out[2] = 0; out[3] = 0;
        }
        return;
    }
    // per entry: feasible machines other than its own; insertion indices in (pred, succ) other than n and n - 1
    int64_t tre = 0, tin = 0;
    for (int n = lane; n < N; n += 32) {
        const int o = row[2 * n], m = row[2 * n + 1];
        const double* tr = ts + (size_t)o * M;
        int f = 0;
        for (int mm = 0; mm < M; ++mm) f += tr[mm] >= 0.0 && mm != m;
        const int j = o % M;
        const int pred = j > 0 ? pos[o - 1] : -1, succ = j < M - 1 ? pos[o + 1] : N;
        int c = succ - pred - 1;
        if (c < 0) c = 0;
        c -= (pred < n && n < succ) + (pred < n - 1 && n - 1 < succ);
        cre[n] = f;
        cin[n] = c;
        tre += f;
        tin += c;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        tre += __shfl_xor_sync(FULL, tre, d);
        tin += __shfl_xor_sync(FULL, tin, d);
    }
    __syncwarp();
    const int64_t R = tre + tin;
    if (R == 0) {
        if (lane == 0) {
            out[0] = (int32_t)q; out[1] = -1; out[2] = 0; out[3] = 0;
        }
        return;
    }
    const int64_t idx = below(u01(A.seed, chain_counter(A.it, k), 0), R);
    const bool ins = idx >= tre;
    int n;
    int64_t r;
    find_entry(ins ? cin : cre, N, ins ? idx - tre : idx, lane, n, r);
    if (lane != 0) return;
    int arg = -1;
    if (n >= 0) {
        const int o = row[2 * n];
        if (!ins) {  // the r-th feasible machine other than the entry's own, in machine order
            const int m = row[2 * n + 1];
            const double* tr = ts + (size_t)o * M;
            for (int mm = 0; mm < M; ++mm) {
                if (tr[mm] >= 0.0 && mm != m && r-- == 0) {
                    arg = mm;
                    break;
                }
            }
        } else {  // the r-th index of (pred, succ) skipping n - 1 and n, in increasing order
            const int j = o % M;
            const int pred = j > 0 ? pos[o - 1] : -1, succ = j < M - 1 ? pos[o + 1] : N;
            int64_t x = pred + 1 + r;
            if (pred < n - 1 && n - 1 < succ && x >= n - 1) ++x;
            if (pred < n && n < succ && x >= n) ++x;
            arg = (int)x;
        }
    }
    out[0] = (int32_t)q;
    out[1] = n >= 0 && arg >= 0 ? (ins ? 1 : 0) : -1;
    out[2] = n >= 0 && arg >= 0 ? n : 0;
    out[3] = n >= 0 && arg >= 0 ? arg : 0;
}

// ---- Metropolis step, exchange and best ------------------------------------------------------------------------------
struct StepArgs {
    int S, N, M, K, it, parity;
    const int32_t *moves, *first_invalid;
    const double *obj, *f4, *temp;
    uint64_t seed;
    int32_t* cur;
    double *cur_obj, *cur_f4;
    int32_t* best;
    double *best_obj, *best_f4;
    int32_t *accepted, *swapped;
};

// one block per instance; its warps loop over the chains, each with a staged copy of the row it rewrites [N,2]
__global__ void __launch_bounds__(MAX_WARPS * 32) anneal_step_kernel(const __grid_constant__ StepArgs A) {
    extern __shared__ int32_t step_smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int s = blockIdx.x, N = A.N, M = A.M, K = A.K;
    int32_t* stage = step_smem + (size_t)w * 2 * N;
    const int64_t q0 = (int64_t)s * K;

    // 1. Metropolis
    for (int k = w; k < K; k += nw) {
        const int64_t q = q0 + k;
        int32_t* cs = A.cur + (size_t)q * N * 2;
        const int32_t* mv = A.moves + q * 4;
        const int row = mv[0], kind = mv[1], ms = mv[2], arg = mv[3];
        int take = 0;
        if (lane == 0) {
            bool ok = row == q && (kind == 0 || kind == 1) && ms >= 0 && ms < N && A.first_invalid[q] == -1;
            if (ok) {
                const int o = cs[2 * ms], mo = cs[2 * ms + 1];
                ok = o >= 0 && o < N && (kind == 0 ? arg >= 0 && arg < M && mo >= 0 && mo < M : arg >= 0 && arg < N);
            }
            const double x = A.obj[q];
            if (ok && x == x) {
                const double delta = x - A.cur_obj[q], T = A.temp[q];
                take = delta <= 0.0 || (T > 0.0 && u01(A.seed, chain_counter(A.it, k), 1) < exp_neg(delta / T));
            }
            A.accepted[q] = take;
            A.swapped[q] = 0;
        }
        take = __shfl_sync(FULL, take, 0);
        if (take) {
            for (int i = lane; i < 2 * N; i += 32) stage[i] = cs[i];
            __syncwarp();
            const bool ins = kind == 1;
            for (int n = lane; n < N; n += 32) {  // search.apply_moves' index arithmetic
                int from = n;
                if (ins) {
                    const int rest = n < arg ? n : n - 1;
                    from = n == arg ? ms : (rest < ms ? rest : rest + 1);
                }
                cs[2 * n] = stage[2 * from];
                cs[2 * n + 1] = !ins && n == ms ? arg : stage[2 * from + 1];
            }
            if (lane < 4) A.cur_f4[q * 4 + lane] = A.f4[q * 4 + lane];
            if (lane == 0) A.cur_obj[q] = A.obj[q];
        }
        __syncwarp();  // the stage is rewritten by the warp's next chain
    }
    __syncthreads();

    // 2. exchange of the pairs (k, k + 1), k = parity (mod 2)
    if (A.parity == 0 || A.parity == 1) {
        for (int k = A.parity + 2 * w; k + 1 < K; k += 2 * nw) {
            const int64_t a = q0 + k, b = a + 1;
            int swap = 0;
            if (lane == 0) {
                const double d = A.cur_obj[b] - A.cur_obj[a], Ta = A.temp[a], Tb = A.temp[b];
                swap = d <= 0.0 ||
                       (Ta > 0.0 && u01(A.seed, chain_counter(A.it, k), 2) < exp_neg(d * (1.0 / Ta - 1.0 / Tb)));
                A.swapped[a] = swap;
            }
            if (__shfl_sync(FULL, swap, 0)) {
                int32_t* ra = A.cur + (size_t)a * N * 2;
                int32_t* rb = A.cur + (size_t)b * N * 2;
                for (int i = lane; i < 2 * N; i += 32) {
                    const int32_t x = ra[i];
                    ra[i] = rb[i];
                    rb[i] = x;
                }
                if (lane < 4) {
                    const double x = A.cur_f4[a * 4 + lane];
                    A.cur_f4[a * 4 + lane] = A.cur_f4[b * 4 + lane];
                    A.cur_f4[b * 4 + lane] = x;
                }
                if (lane == 0) {
                    const double x = A.cur_obj[a];
                    A.cur_obj[a] = A.cur_obj[b];
                    A.cur_obj[b] = x;
                }
            }
        }
    }
    __syncthreads();

    // 3. best: the least cur_obj strictly below best_obj, ties to the lowest k; NaN never wins
    if (w != 0) return;
    double v = A.best_obj[s];
    int bk = -1;
    for (int k = lane; k < K; k += 32) {
        const double x = A.cur_obj[q0 + k];
        if (x < v) {
            v = x;
            bk = k;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const double v2 = __shfl_xor_sync(FULL, v, d);
        const int b2 = __shfl_xor_sync(FULL, bk, d);
        if (b2 >= 0 && (bk < 0 || v2 < v || (v2 == v && b2 < bk))) {
            v = v2;
            bk = b2;
        }
    }
    if (bk < 0) return;
    const int64_t q = q0 + bk;
    const int32_t* cs = A.cur + (size_t)q * N * 2;
    int32_t* bs = A.best + (size_t)s * N * 2;
    for (int i = lane; i < 2 * N; i += 32) bs[i] = cs[i];
    if (lane < 4) A.best_f4[(size_t)s * 4 + lane] = A.cur_f4[q * 4 + lane];
    if (lane == 0) A.best_obj[s] = v;
}

// warps per block: as many of `per_warp` bytes as fit in 48 KB, at most MAX_WARPS
int warps_for(size_t per_warp) {
    const size_t w = (48 * 1024) / per_warp;
    return w < 1 ? 1 : (w > MAX_WARPS ? MAX_WARPS : (int)w);
}

bool bad_size(int S, int J, int M, int K) {
    return S < 1 || K < 1 || J < 1 || M < 2 || M > 64 || (int64_t)J * M > 4096 || (int64_t)S * K > INT32_MAX;
}

}  // namespace

extern "C" {

int mtfjsp_anneal_propose(const double* t, int S, int J, int M, int K, const int32_t* cur, uint64_t seed, int it,
                          int32_t* moves, void* stream) {
    if (!t || !cur || !moves || bad_size(S, J, M, K) || it < 0)
        return fail(MTFJSP_E_ARG, "mtfjsp_anneal_propose: bad argument");
    ProposeArgs A;
    A.t = t; A.S = S; A.N = J * M; A.M = M; A.K = K; A.it = it; A.Q = (int64_t)S * K;
    A.cur = cur; A.seed = seed; A.moves = moves;
    const int wpb = warps_for(propose_warp_bytes(A.N));  // 3 * 4096 * 4 B = 48 KB at most: no opt-in
    const unsigned grid = (unsigned)((A.Q + wpb - 1) / wpb);
    anneal_propose_kernel<<<grid, wpb * 32, wpb * propose_warp_bytes(A.N), (cudaStream_t)stream>>>(A);
    return launched(__func__);
}

int mtfjsp_anneal_step(int S, int J, int M, int K, const int32_t* moves, const int32_t* first_invalid,
                       const double* obj, const double* f4, const double* temp, uint64_t seed, int it, int swap_parity,
                       int32_t* cur, double* cur_obj, double* cur_f4, int32_t* best, double* best_obj, double* best_f4,
                       int32_t* accepted, int32_t* swapped, void* stream) {
    if (!moves || !first_invalid || !obj || !f4 || !temp || !cur || !cur_obj || !cur_f4 || !best || !best_obj ||
        !best_f4 || !accepted || !swapped || bad_size(S, J, M, K) || it < 0)
        return fail(MTFJSP_E_ARG, "mtfjsp_anneal_step: bad argument");
    StepArgs A;
    A.S = S; A.N = J * M; A.M = M; A.K = K; A.it = it; A.parity = swap_parity;
    A.moves = moves; A.first_invalid = first_invalid; A.obj = obj; A.f4 = f4; A.temp = temp; A.seed = seed;
    A.cur = cur; A.cur_obj = cur_obj; A.cur_f4 = cur_f4;
    A.best = best; A.best_obj = best_obj; A.best_f4 = best_f4;
    A.accepted = accepted; A.swapped = swapped;
    const size_t per_warp = (size_t)A.N * 2 * sizeof(int32_t);
    int wpb = warps_for(per_warp);
    if (wpb > K) wpb = K;
    anneal_step_kernel<<<S, wpb * 32, wpb * per_warp, (cudaStream_t)stream>>>(A);
    return launched(__func__);
}

}  // extern "C"
