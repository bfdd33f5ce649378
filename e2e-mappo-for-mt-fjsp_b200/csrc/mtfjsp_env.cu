// mtfjsp_env.cu -- batched MT-FJSP disjunctive-graph environment for sm_100a (B200).
//
// Two kernels share one algorithm.  env_kernel: one warp per environment, run-time sizes (reset, and sizes without a
// specialisation).  env_kernel_s: compile-time (J, M), G lanes per environment and 32/G environments per warp -- the
// hot kernel.  Per launch a lane group stages its instance's records from HBM into shared memory (one TMA bulk copy per
// record), draws the random action itself when asked to (MODE_POLICY: random-rollout step in one launch), applies the
// (operation, machine) action, recomputes the reward, rewrites the observation rows the step changed (or all of them)
// and writes back only the state words that changed.
//
// What this replaces in the reference (file:line, "SS" = graph-jsp-env/src/graph_jsp_env/
// disjunctive_graph_jsp_env_singlestep.py):
//   transition      SS:716-974, 1476-1809; trainer/DGenv_func.py:46-170
//   reward          SS:1051-1171           reward scaling  algorithm/ppo_trick.py:54-122
//   observation     SS:1920-2515           job mask        algorithm/ppo_algorithm.py:202-317
//   machine feats   trainer/parallel_env.py:152-214
//
// Numerics: all schedule arithmetic is FP64 in the reference's operand order; this file must be
// compiled with -fmad=false (no FMA contraction).  np.sum is restated as numpy's pairwise summation
// (8 accumulators, 128-element leaves) so that energy totals are bit-identical.
//
// HBM layout (per handle, B environments; every record is 16-byte aligned):
//   sd  [B][sd_stride] f64   dynamic doubles: st[N] ft[N] dur[N] psel[N] | mk_prev e_prev trans idle_prev |
//                            macc[M][3] | w[3] | eacc[L][8] eleaf[L] ipre[C] | scaler R[4] mean[4] S[4] n
//                            (for an unscheduled op st/ft hold the current estimate, dur = 0, psel = min energy;
//                            eacc / eleaf cache numpy's pairwise summation of the energy estimate: the 8 accumulators
//                            and the result of each of its L leaves, so a step re-adds one accumulator chain only;
//                            ipre (N > 128 only, C = ceil(N/32)) caches the running idle-time sum in front of every
//                            32nd term of the flat order: a step re-adds from the chunk it inserted into)
//   si  [B][si_stride] i16   dynamic ints:    mach[N] ord[N] rpred[N] cnt[M] | removed_head fresh_co nsched | nxt[J]
//                            (ord = the scheduled ops in (machine, route position) order: machine m's route is
//                            ord[off_m, off_m + cnt[m]) with off_m = cnt[0] + ... + cnt[m-1]; rpred = route predecessor)
//   xs  [B][xs_stride] f64   static doubles:  mind[N] minpt[N] tt[M][M]
//   t,p [B][N][M]      f64   instance tables, touched only at (op, machine) and in the mfea1 kernel
#include <assert.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/mtfjsp.h"

#define MAX_LEAVES 64
#define MAX_PROG 128
#define FULL 0xffffffffu

namespace {

struct Layout {
    int B, J, M, N, E, left_shift;
    int sd_stride, si_stride, xs_stride;
    int o_st, o_ft, o_dur, o_psel, o_scal, o_macc, o_w, o_eacc, o_eleaf, o_ipre, nich, o_sc;  // sd offsets (doubles)
    int o_mach, o_ord, o_rpred, o_cnt, o_misc, o_nxt;          // si offsets (int16)
    int o_mind, o_minpt, o_tt;                                 // xs offsets (doubles)
    int sm_sd, sm_xs, sm_pt, sm_v, sm_leaf, sm_si, sm_off, sm_nxt, sm_tail;  // smem byte offsets per warp
    int smem_per_warp, warps_per_block;
};

struct PwPlan {  // numpy pairwise-sum plan for N elements
    int nleaves, nprog;
    int leaf_off[MAX_LEAVES];
    int leaf_len[MAX_LEAVES];
    signed char prog[MAX_PROG];  // postfix: k >= 0 push leaf k, -1 add
};

struct Params {
    Layout L;
    PwPlan pw;
    double* sd;
    int16_t* si;
    const double* xs;
    const double* t;
    const double* p;
    const double* weights;  // reset, and MODE_FROM_RESET
    // MODE_FROM_RESET: the step also performs a recorded episode reset (mtfjsp_env::pend_reset): the records are staged
    // from the snapshot sd0 / si0, the weights from `weights`, the reward scaler's running returns cleared if clear_ret,
    // and the records written back whole
    const double* sd0;
    const int16_t* si0;
    int clear_ret;
    double cfgw[3], divisor, gamma;
    // step io
    const int32_t* op;
    const int32_t* mach;
    double* reward5;
    double* scaled4;
    uint8_t* done;
    uint8_t* invalid;
    double* info6;  // optional [B,6] = (r, done, mk_s, idle_s, pt_s, tt_s), trainer/parallel_env.py:260
    const int2* act2;      // optional packed actions [B] (op, machine); used instead of op / mach when set
    // MODE_POLICY (random-rollout step): the counter-based random valid action is drawn in the kernel from the masks the
    // previous launch left in jm_* / cand_int, and the candidate-machine features of the drawn op are written
    uint64_t seed, env_offset;
    const int8_t* edge_id;
    int32_t* op_out;
    int32_t* mach_out;
    void* mfea1;     // [B,M,6] OutT or NULL
    uint8_t* mmask;  // [B,M] or NULL
    unsigned char* rec;    // optional packed step records, rec_stride bytes per env (include/mtfjsp.h, mtfjsp_step_host_packed):
                           // f64 r | f64 scaled[4] | u8 done | u8 mask_bits[ceil(J/8)] | u8 next_op[J] | padding to 8
    int rec_stride;
    int rev;        // blocks walk the env range from its END (alternate launches: what the previous launch touched last is
                    // still in L2 when this one starts -- a batch's working set is larger than the 126 MB L2, and a
                    // forward walk every launch evicts each line just before it is needed again)
    // obs io
    void* tfea;
    void* mfea;
    float* adj_w;
    int16_t* adj_src;
    uint8_t* jmask;
    int32_t* cand;
    int mask_mode;
    int obs_inc;  // fused step+obs only: the output buffers hold the previous observation, rewrite just the rows that changed
    // always-written internal mask / candidate buffers (policy kernel, host step)
    uint8_t* jm_fin;
    uint8_t* jm_esa;
    int32_t* cand_int;
    // launch overlap (size-specialised whole-batch step launches, see ovl_wait): ep != 0 makes each warp release
    // done_ep[its env range] = ep once its envs are written; wait_ep != 0 makes each warp first wait until that entry
    // reaches wait_ep (the previous such launch may still be running); ovl_err: mapped host word set on a timeout
    unsigned long long* done_ep;
    unsigned long long ep, wait_ep;
    unsigned* ovl_err;
};

enum { MODE_STEP = 1, MODE_OBS = 2, MODE_RESET = 4, MODE_POLICY = 8,
       MODE_HOST = 16,        // size-specialised kernels: step info / packed records leave as whole-warp runs (host-step calls)
       MODE_FROM_RESET = 32 };  // size-specialised step kernels: the step also performs a recorded reset (Params::sd0)

// step info (r, done, mk_s, idle_s, pt_s, tt_s) goes to the contiguous [B,6] array and / or the packed host record
#define INFO6_PUT(b_, k_, v_)                                                                               \
    do {                                                                                                    \
        if (P.info6) P.info6[(size_t)(b_) * 6 + (k_)] = (v_);                                               \
        if (P.rec) {                                                                                        \
            unsigned char* r_ = P.rec + (size_t)(b_) * P.rec_stride;                                        \
            if ((k_) == 1) r_[REC_DONE] = (v_) != 0.0 ? 1 : 0;                                              \
            else reinterpret_cast<double*>(r_)[(k_) == 0 ? 0 : (k_) - 1] = (v_);                            \
        }                                                                                                   \
    } while (0)
// packed record: f64 r @0, f64 scaled[4] @8, u8 done @40, u8 mask_bits[ceil(J/8)] @41, u8 next_op[J] behind them
constexpr int REC_DONE = 40, REC_BITS = 41;
__host__ __device__ constexpr int rec_bytes(int J) { return (REC_BITS + (J + 7) / 8 + J + 7) / 8 * 8; }

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

// adjacency value of an arc with weight w leaving op u (SS:2019, 2050-2064); 0 = arc vanishes
__device__ __forceinline__ double adj_val(double w, bool u_assigned, double dur_u) {
    long long wi = (long long)w;
    if (wi == 0) return 0.0;
    double nd = u_assigned ? dur_u : 1.0;
    long long v = (long long)((double)wi - nd);
    return (double)(v + 1);
}

template <typename OutT>
__device__ __forceinline__ void store_row(OutT* dst, const double* f, int n);
template <>
__device__ __forceinline__ void store_row<float>(float* dst, const double* f, int n) {
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int k = 0; k < n / 4; k++)
        d4[k] = make_float4((float)f[4 * k], (float)f[4 * k + 1], (float)f[4 * k + 2], (float)f[4 * k + 3]);
}
template <>
__device__ __forceinline__ void store_row<double>(double* dst, const double* f, int n) {
    double2* d2 = reinterpret_cast<double2*>(dst);
    for (int k = 0; k < n / 2; k++) d2[k] = make_double2(f[2 * k], f[2 * k + 1]);
}

// numpy pairwise sum of a[0..N) following the host-built plan; every lane returns the result.  eacc [nleaves][8] / eleaf
// [nleaves] receive the 8 accumulators (before their tree) and the result of every leaf: the cache the size-specialised
// kernel updates incrementally (one accumulator chain per step).
__device__ double pairwise_sum(const double* a, const PwPlan& pw, double* s_leaf, int lane, double* eacc, double* eleaf) {
    const int grp = lane >> 3, k = lane & 7;
    for (int L0 = 0; L0 < pw.nleaves; L0 += 4) {
        int Lx = L0 + grp;
        bool act = Lx < pw.nleaves;
        int off = act ? pw.leaf_off[Lx] : 0, n = act ? pw.leaf_len[Lx] : 0;
        const int nb = (n >= 8) ? n - (n & 7) : 0;
        double r = 0.0;
        if (n >= 8) {
            r = a[off + k];
            for (int i = 8 + k; i < nb; i += 8) r += a[off + i];
            if (act) eacc[Lx * 8 + k] = r;
        }
        // ((r0+r1)+(r2+r3)) + ((r4+r5)+(r6+r7)); every lane takes part in the shuffles
        r = r + __shfl_down_sync(FULL, r, 1, 8);
        r = r + __shfl_down_sync(FULL, r, 2, 8);
        r = r + __shfl_down_sync(FULL, r, 4, 8);
        double res = r;  // n < 8 (only when N < 8): r is 0 and the loop below is the plain sum
        if (k == 0)
            for (int i = nb; i < n; i++) res += a[off + i];
        if (act && k == 0) { s_leaf[Lx] = res; if (pw.nleaves > 1) eleaf[Lx] = res; }
    }
    __syncwarp();
    if (pw.nleaves == 1) return s_leaf[0];
    // combine leaves with the recursion's shape (postfix program); stack lives above the leaves
    double* stk = s_leaf + MAX_LEAVES;
    int sp = 0;
    double top = 0.0;
    for (int i = 0; i < pw.nprog; i++) {
        int c = pw.prog[i];
        if (c >= 0) {
            if (lane == 0) stk[sp] = s_leaf[c];
            sp++;
        } else {
            __syncwarp();
            double x = stk[sp - 2], y = stk[sp - 1];
            __syncwarp();
            top = x + y;
            sp--;
            if (lane == 0) stk[sp - 1] = top;
        }
        __syncwarp();
    }
    return top;
}

// One env's records staged in shared memory at the Layout::sm_* offsets of its warp's slice `base`: the state the generic
// kernel steps (env_kernel) and the replay kernel runs whole episodes on (replay_kernel)
struct EnvSmem {
    double *sd, *xs, *pt, *v, *leaf;
    int16_t *si, *nxt;
    double *st, *ft, *dur, *psel, *scal, *macc, *ipre, *eacc, *eleaf;
    int16_t *mach, *ord, *rpred, *cnt, *misc;
    const double *mind, *minpt, *tt;
    __device__ __forceinline__ EnvSmem(const Layout& L, unsigned char* base) {
        sd = reinterpret_cast<double*>(base + L.sm_sd);
        xs = reinterpret_cast<double*>(base + L.sm_xs);
        pt = reinterpret_cast<double*>(base + L.sm_pt);  // idle terms, then est_pt
        v = reinterpret_cast<double*>(base + L.sm_v);    // per-job ESA key
        leaf = reinterpret_cast<double*>(base + L.sm_leaf);
        si = reinterpret_cast<int16_t*>(base + L.sm_si);
        nxt = reinterpret_cast<int16_t*>(base + L.sm_nxt);
        st = sd + L.o_st; ft = sd + L.o_ft; dur = sd + L.o_dur; psel = sd + L.o_psel;
        scal = sd + L.o_scal;  // mk_prev, e_prev, trans, idle_prev
        macc = sd + L.o_macc; ipre = sd + L.o_ipre; eacc = sd + L.o_eacc; eleaf = sd + L.o_eleaf;
        mach = si + L.o_mach; ord = si + L.o_ord; rpred = si + L.o_rpred; cnt = si + L.o_cnt;
        misc = si + L.o_misc;  // removed_head, fresh_co, nsched
        mind = xs + L.o_mind; minpt = xs + L.o_minpt; tt = xs + L.o_tt;
    }
};

// The transition's pieces on raw views of the records, shared by the generic step (env_transition, env_estimates,
// env_reward: env_kernel, replay_kernel) and the one-step lookahead (peek_kernel), whose shared-memory layout differs.

// term g of the flat-order idle-time sum (DGenv_func.py:144-170): the gap in front of op ord[g] on its machine
__device__ __forceinline__ double idle_term(const double* st, const double* ft, const int16_t* ord, const int16_t* rpred,
                                            int g) {
    const int v = ord[g], rp = rpred[v];
    return (rp < 0) ? (st[v] - 0.0) : (st[v] - ft[rp]);
}

// op v's term of the energy estimate (SS:896): scheduled ? duration * energy rate : minimum energy
__device__ __forceinline__ double energy_est(const int16_t* mach, const double* dur, const double* psel,
                                             const double* minpt, int v) {
    return (mach[v] >= 0) ? dur[v] * psel[v] : minpt[v];
}

// step reward of a valid transition (wrk_reward_function, SS:1066-1132) from the previous-step scalars scal = (mk_prev,
// e_prev, trans_prev, idle_prev) and the step's makespan estimate mkv, energy estimate env, transport and idle sums:
// (total before the divisor, r_mk, r_idle, r_pt, r_tt)
struct StepReward {
    double total, r_t, r_idle, r_pt, r_tt;
};
__device__ __forceinline__ StepReward reward_terms(const double* scal, const double* cfgw, int N, double mkv, double env,
                                                   double trans, double idle) {
    const double mk_prev = scal[0], e_prev = scal[1], trans_prev = scal[2], idle_prev = scal[3];
    StepReward w;
    w.r_t = 1.0 * mk_prev - mkv;
    double r_pt = 1.0 * e_prev - env;
    w.r_pt = r_pt / (double)N;
    w.r_tt = 1.0 * trans_prev - trans;
    w.r_idle = 1.0 * idle_prev - idle;
    w.total = cfgw[0] * w.r_t + cfgw[1] * (w.r_pt + 1.0 * w.r_idle) + cfgw[2] * w.r_tt * 1.0;
    return w;
}

// what one transition leaves for the step's reward epilogue and incremental observation
struct StepOut {
    bool valid, done;
    double idle, nt, trans, ec;
    int o_next, o_tail;  // machine follower and route tail of the stepped op
};

// One transition of action (a, m) on the staged env (SS:716-974, 1476-1809; trainer/DGenv_func.py:46-170): validity,
// placement with or without left shift, the move into the flat order, the flat-order idle-time sum and the step's
// transport and energy terms.  tp: the env's row of the instance tables t / p.  WB: also write what changed to the env's
// records g_sd / g_si (the generic step kernel); the replay kernel runs on the staged copy only.
template <bool WB>
__device__ __forceinline__ StepOut env_transition(const Layout& L, const EnvSmem& S, const double* t, const double* p,
                                                  size_t tp, int a, int m, double* g_sd, int16_t* g_si, int lane) {
    const int N = L.N, M = L.M;
    StepOut o;
    o.valid = false; o.done = false; o.idle = 0.0; o.nt = 0.0; o.trans = 0.0; o.ec = 0.0; o.o_next = -1; o.o_tail = -1;
    const int nsched0 = S.misc[2];
    double d = 0.0, pa = 0.0;
    bool valid = (a >= 0) && (a < N) && (m >= 0) && (m < M) && (nsched0 < N);
    if (valid) valid = (S.mach[a] < 0) && (((a % M) == 0) || (S.mach[a - 1] >= 0));
    if (valid) {
        d = __ldg(t + (tp * N + a) * M + m);
        pa = __ldg(p + (tp * N + a) * M + m);
        valid = !(d < 0);
    }
    o.valid = valid;
    if (valid) {
        const bool first = (a % M) == 0;
        const int ja = a / M;
        // job-arc refresh at step start (SS:1502): transient markers of the previous step expire
        int rem_head = -1, fresh = -1;
        const double arr_a = first ? 0.0 : S.ft[a - 1] + S.tt[S.mach[a - 1] * M + m];  // DGenv_func.py:46-66
        const int len = S.cnt[m];
        const double ttmm = S.tt[m * M + m];
        double st = arr_a;
        int where = 0, prev = -1, next = -1;
        // machine m's route is ord[offm, offm + len)
        int offm = 0;
        for (int m0 = 0; m0 < m; m0 += 32) offm += __reduce_add_sync(FULL, (m0 + lane < m) ? (int)S.cnt[m0 + lane] : 0);
        if (len > 0) {
            // one pass over the route of machine m: arrival of each op, first feasible slot (SS:1548-1601)
            const double lbft = arr_a + d;
            unsigned best = 0xffffffffu;
            const int lastop = S.ord[offm + len - 1];
            if (L.left_shift) {
                for (int k0 = 0; k0 < len; k0 += 32) {
                    const int k = k0 + lane;
                    unsigned key = 0xffffffffu;
                    if (k < len) {
                        const int v = S.ord[offm + k];
                        const bool vfirst = (v % M) == 0;
                        double nst = vfirst ? 0.0 : S.ft[v - 1] + S.tt[S.mach[v - 1] * M + m];
                        bool ok;
                        if (k == 0) {
                            ok = (lbft <= nst);  // SS:1548 (route head has no machine in-arc)
                        } else {
                            const int rp = S.ord[offm + k - 1];
                            double val = S.ft[rp] + ((rp / M == v / M) ? ttmm : 0.0);
                            nst = fmax(nst, val);
                            ok = !(lbft > nst) && !((nst - S.ft[rp]) < d);  // SS:1597-1601
                        }
                        if (ok) key = ((unsigned)k << 16) | (unsigned)v;
                    }
                    best = min(best, __reduce_min_sync(FULL, key));
                }
            }
            if (best != 0xffffffffu) {
                where = (int)(best >> 16);
                next = (int)(best & 0xffffu);
                if (where > 0) {
                    prev = S.rpred[next];
                    double y = S.ft[prev] + ((prev / M == ja) ? ttmm : 0.0);  // SS:1619
                    st = (y > arr_a) ? y : arr_a;
                    if (next == prev + 1 && (next % M) != 0) rem_head = next;  // SS:1660
                }
            } else {  // _append_at_the_end, SS:1689-1775
                where = len;
                prev = lastop;
                double y = S.ft[prev] + ((prev / M == ja) ? ttmm : 0.0);
                st = (y > arr_a) ? y : arr_a;
            }
            if (prev >= 0 && prev == a - 1 && !first) fresh = a;
            o.o_tail = (where == len) ? a : lastop;
        } else {
            o.o_tail = a;
        }
        o.o_next = next;
        __syncwarp();
        // ---- apply: open slot p of the flat order (entries behind it move up by one), link the op in ----
        const int p_ = offm + where;
        for (int g0 = ((nsched0 > 0 ? nsched0 - 1 : 0) / 32) * 32; g0 >= 0 && g0 + 31 >= p_; g0 -= 32) {
            const int g = g0 + lane;
            const bool mv_ = g >= p_ && g < nsched0;
            const int16_t x = mv_ ? S.ord[g] : (int16_t)0;
            __syncwarp();
            if (mv_) {
                S.ord[g + 1] = x;
                if (WB) g_si[L.o_ord + g + 1] = x;
            }
            __syncwarp();
        }
        if (lane == 0) {
            S.mach[a] = (int16_t)m; S.ord[p_] = (int16_t)a; S.rpred[a] = (int16_t)prev;
            if (next >= 0) S.rpred[next] = (int16_t)a;
            S.cnt[m] = (int16_t)(len + 1);
            S.misc[0] = (int16_t)rem_head; S.misc[1] = (int16_t)fresh; S.misc[2] = (int16_t)(nsched0 + 1);
            S.st[a] = st; S.ft[a] = st + d; S.dur[a] = d; S.psel[a] = pa;
            if (WB) {
                g_si[L.o_mach + a] = (int16_t)m; g_si[L.o_ord + p_] = (int16_t)a; g_si[L.o_rpred + a] = (int16_t)prev;
                if (next >= 0) g_si[L.o_rpred + next] = (int16_t)a;
                g_si[L.o_cnt + m] = (int16_t)(len + 1);
                g_si[L.o_misc + 0] = (int16_t)rem_head; g_si[L.o_misc + 1] = (int16_t)fresh;
                g_si[L.o_misc + 2] = (int16_t)(nsched0 + 1);
                g_si[L.o_nxt + ja] = (int16_t)((a % M) + 1);
                g_sd[L.o_st + a] = st; g_sd[L.o_ft + a] = st + d; g_sd[L.o_dur + a] = d; g_sd[L.o_psel + a] = pa;
                double cur = st + d;  // estimator chain of the remaining ops of this job (SS:1964-1995)
                for (int c = (a % M) + 1; c < M; c++) {
                    g_sd[L.o_st + ja * M + c] = cur;
                    cur = cur + S.mind[ja * M + c];
                    g_sd[L.o_ft + ja * M + c] = cur;
                }
            }
        }
        __syncwarp();
        const int nsched = nsched0 + 1;
        o.done = (nsched == N);
        // ---- idle time: sequential sum in (machine, route) order = flat order, DGenv_func.py:144-170 ----
        for (int g = lane; g < nsched; g += 32) S.pt[g] = idle_term(S.st, S.ft, S.ord, S.rpred, g) * 1.0;
        __syncwarp();
        double idle = 0.0;
        if (L.nich) {  // large instances: running sum in front of every 32nd term (the specialised kernel restarts there)
            for (int g = 0; g <= nsched; g++) {
                if ((g & 31) == 0 && (g >> 5) < L.nich && lane == 0) S.ipre[g >> 5] = idle;
                if (g < nsched) idle = idle + S.pt[g];
            }
        } else {
#pragma unroll 4
            for (int g = 0; g < nsched; g++) idle = idle + S.pt[g];
        }
        __syncwarp();
        o.idle = idle;
        o.nt = first ? 0.0 : S.tt[S.mach[a - 1] * M + m];  // SS:872-877
        o.trans = S.scal[2] + o.nt;
        o.ec = pa * d;
    }
    __syncwarp();
    return o;
}

// Per-job walk over the staged env: scheduled prefix, estimator chain (SS:1964-1995), ESA key (ppo_algorithm.py:280),
// est_pt; with SUMS the makespan estimate (*mkv) and the energy estimate (*env, numpy's pairwise sum) (SS:894-896)
template <bool SUMS>
__device__ __forceinline__ void env_estimates(const Layout& L, const PwPlan& pw, const EnvSmem& S, int lane, double* mkv,
                                              double* env) {
    const int N = L.N, M = L.M, J = L.J;
    for (int j = lane; j < J; j += 32) {
        const int jb = j * M;
        double cur = 0.0, rm = 0.0;
        int nx = 0;
        while (nx < M && S.mach[jb + nx] >= 0) {
            cur = S.ft[jb + nx];
            rm = fmax(rm, cur);
            nx++;
        }
        for (int c = nx; c < M; c++) {
            S.st[jb + c] = (c == 0) ? 0.0 : cur;
            cur = ((c == 0) ? 0.0 : cur) + S.mind[jb + c];
            S.ft[jb + c] = cur;
        }
        S.nxt[j] = (int16_t)nx;
        S.v[j] = (nx == M) ? INFINITY : rm;
    }
    __syncwarp();
    double mx = -INFINITY;
    for (int v = lane; v < N; v += 32) {
        S.pt[v] = energy_est(S.mach, S.dur, S.psel, S.minpt, v);
        mx = fmax(mx, S.ft[v]);
    }
    __syncwarp();
    if (SUMS) {
        *mkv = warp_max(mx);
        *env = pairwise_sum(S.pt, pw, S.leaf, lane, S.eacc, S.eleaf);
    }
}

// step reward of a valid transition (reward_terms); lane 0 then advances the machine accumulators (SS:2323-2338) and the
// previous-step scalars (SS:932-936)
__device__ __forceinline__ StepReward env_reward(const Layout& L, const EnvSmem& S, const double* cfgw, int m, double mkv,
                                                 double env, const StepOut& o, int lane) {
    const int N = L.N;
    const StepReward w = reward_terms(S.scal, cfgw, N, mkv, env, o.trans, o.idle);
    const double idle_prev = S.scal[3];  // read after reward_terms: the scalar loads keep their order in the SASS
    __syncwarp();
    if (lane == 0) {
        S.macc[m * 3 + 0] += o.ec / (double)N;
        S.macc[m * 3 + 1] += o.nt;
        S.macc[m * 3 + 2] += o.idle - idle_prev;
        S.scal[0] = mkv; S.scal[1] = env; S.scal[2] = o.trans; S.scal[3] = o.idle;
    }
    return w;
}

template <int MODE, typename OutT>
__global__ void __launch_bounds__(256) env_kernel(const __grid_constant__ Params P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Layout& L = P.L;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * L.warps_per_block + warp;
    if (b >= L.B) return;
    const int N = L.N, M = L.M, J = L.J;
    unsigned char* base = smem_raw + (size_t)warp * L.smem_per_warp;
    const EnvSmem S(L, base);
    double* s_sd = S.sd;
    double* s_xs = S.xs;
    double* s_pt = S.pt;
    double* s_v = S.v;
    int16_t* s_si = S.si;
    int16_t* s_nxt = S.nxt;
    int16_t* s_tail = reinterpret_cast<int16_t*>(base + L.sm_tail);

    double* g_sd = P.sd + (size_t)b * L.sd_stride;
    int16_t* g_si = P.si + (size_t)b * L.si_stride;
    const double* g_xs = P.xs + (size_t)b * L.xs_stride;

    // ---- stage records (128-bit, coalesced) ----
    {
        const uint4* src = reinterpret_cast<const uint4*>(g_sd);
        uint4* dst = reinterpret_cast<uint4*>(s_sd);
        for (int i = lane; i < L.sd_stride / 2; i += 32) dst[i] = src[i];
        src = reinterpret_cast<const uint4*>(g_xs);
        dst = reinterpret_cast<uint4*>(s_xs);
        for (int i = lane; i < L.xs_stride / 2; i += 32) dst[i] = __ldg(src + i);
        if (!(MODE & MODE_RESET)) {
            src = reinterpret_cast<const uint4*>(g_si);
            dst = reinterpret_cast<uint4*>(s_si);
            for (int i = lane; i < L.si_stride / 8; i += 32) dst[i] = src[i];
        }
    }
    double* s_st = S.st;
    double* s_ft = S.ft;
    double* s_dur = S.dur;
    double* s_psel = S.psel;
    double* s_scal = S.scal;
    double* s_macc = S.macc;
    double* s_w = s_sd + L.o_w;
    double* s_sc = s_sd + L.o_sc;  // R[4] mean[4] S[4] n
    int16_t* s_mach = S.mach;
    int16_t* s_ord = S.ord;
    int16_t* s_rpred = S.rpred;
    int16_t* s_cnt = S.cnt;
    int16_t* s_misc = S.misc;
    const double* s_minpt = S.minpt;
    const double* s_tt = S.tt;

    if (MODE & MODE_RESET) {  // load_instance + reset, SS:397-714, 1183-1245
        __syncwarp();
        for (int i = lane; i < 4 * N; i += 32) s_sd[L.o_st + i] = 0.0;  // st ft dur psel are contiguous
        for (int i = lane; i < 3 * M; i += 32) s_macc[i] = 0.0;
        for (int i = L.o_eacc + lane; i < L.o_sc; i += 32) s_sd[i] = 0.0;
        if (lane < 3) s_w[lane] = P.weights[(size_t)b * 3 + lane];
        if (lane < 4) s_scal[lane] = 0.0;
        for (int i = lane; i < N; i += 32) { s_mach[i] = -1; s_ord[i] = -1; s_rpred[i] = -1; }
        for (int i = lane; i < M; i += 32) s_cnt[i] = 0;
        if (lane == 0) { s_misc[0] = -1; s_misc[1] = -1; s_misc[2] = 0; }
        for (int i = L.o_misc + 3 + lane; i < L.si_stride; i += 32) s_si[i] = 0;
    }
    __syncwarp();

    int a = -1, m = -1;
    double mkv = 0.0, env = 0.0;
    StepOut so;  // step results kept in registers for the reward epilogue and the incremental observation
    so.valid = false; so.done = false; so.o_next = -1; so.o_tail = -1;
    // incremental observation (see env_kernel_s): previous transients
    int rem_prev = -1, fresh_prev = -1;

    if (MODE & MODE_STEP) {
        if (P.act2) { const int2 am = P.act2[b]; a = am.x; m = am.y; }
        else { a = P.op[b]; m = P.mach[b]; }
        rem_prev = s_misc[0];
        fresh_prev = s_misc[1];
        so = env_transition<true>(L, S, P.t, P.p, (size_t)b, a, m, g_sd, g_si, lane);
    }
    const bool valid = so.valid, done = so.done;
    const int o_next = so.o_next, o_tail = so.o_tail;

    env_estimates<(MODE & (MODE_STEP | MODE_RESET)) != 0>(L, P.pw, S, lane, &mkv, &env);

    if (MODE & MODE_RESET) {
        if (lane == 0) { s_scal[0] = mkv; s_scal[1] = env; s_scal[2] = 0.0; s_scal[3] = 0.0; }  // SS:697-705
        __syncwarp();
        // write back the env part of sd (everything except the scaler block) and the whole si record.
        // State invariant: an unscheduled op carries its estimate in st/ft, dur = 0 and psel = min energy.
        for (int i = lane; i < N; i += 32) {
            g_sd[L.o_st + i] = s_st[i];
            g_sd[L.o_ft + i] = s_ft[i];
            g_sd[L.o_dur + i] = 0.0;
            g_sd[L.o_psel + i] = s_minpt[i];
        }
        for (int i = L.o_scal + lane; i < L.o_sc; i += 32) g_sd[i] = s_sd[i];
        uint4* dst = reinterpret_cast<uint4*>(g_si);
        const uint4* src = reinterpret_cast<const uint4*>(s_si);
        for (int i = lane; i < L.si_stride / 8; i += 32) dst[i] = src[i];
    }

    if ((MODE & MODE_STEP)) {
        if (valid) {
            const StepReward rw = env_reward(L, S, P.cfgw, m, mkv, env, so, lane);
            const double r_t = rw.r_t, r_idle = rw.r_idle, r_pt = rw.r_pt, r_tt = rw.r_tt, total = rw.total;
            // reward scaling, ppo_trick.py:73-88,115-119 (lanes 0..3 own one component each)
            double scaled = 0.0;
            if (lane < 4) {
                const double x = lane == 0 ? r_t : lane == 1 ? r_idle : lane == 2 ? r_pt : r_tt;  // parallel_env.py:255
                double R = P.gamma * s_sc[lane] + x;
                double nn = s_sc[12] + 1.0;
                double mean, S = s_sc[8 + lane], sd_;
                if (nn == 1.0) {
                    mean = R;
                    sd_ = fabs(R);
                } else {
                    double old = s_sc[4 + lane];
                    mean = old + (R - old) / nn;
                    S = S + (R - old) * (R - mean);
                    sd_ = sqrt(S / nn);
                }
                scaled = x / (sd_ + 1e-8);
                __syncwarp(0xf);
                s_sc[lane] = R; s_sc[4 + lane] = mean; s_sc[8 + lane] = S;
                if (lane == 0) s_sc[12] = nn;
                if (P.scaled4) P.scaled4[(size_t)b * 4 + lane] = scaled;
                INFO6_PUT(b, 2 + lane, scaled);
            }
            __syncwarp();
            // selective write-back of the doubles that changed: scalars, macc[m], scaler
            if (lane < 20) {
                int idx = lane < 4 ? L.o_scal + lane : lane < 7 ? L.o_macc + m * 3 + (lane - 4) : L.o_sc + (lane - 7);
                g_sd[idx] = s_sd[idx];
            }
            for (int i = L.o_eacc + lane; i < L.o_sc; i += 32) g_sd[i] = s_sd[i];  // energy-sum cache (this kernel recomputes all of it)
            if (lane == 0) {
                if (P.reward5) {
                    double* r5 = P.reward5 + (size_t)b * 5;
                    r5[0] = total / P.divisor; r5[1] = r_t; r5[2] = r_idle; r5[3] = r_pt; r5[4] = r_tt;
                }
                if (P.done) P.done[b] = done ? 1 : 0;
                if (P.invalid) P.invalid[b] = 0;
                INFO6_PUT(b, 0, total / P.divisor); INFO6_PUT(b, 1, done ? 1.0 : 0.0);
            }
        } else {
            if (lane < 5 && P.reward5) P.reward5[(size_t)b * 5 + lane] = 0.0;
            if (lane < 4 && P.scaled4) P.scaled4[(size_t)b * 4 + lane] = 0.0;
            if (lane < 6 && lane != 1) INFO6_PUT(b, lane, 0.0);
            if (lane == 0) {
                if (P.done) P.done[b] = (s_misc[2] == N) ? 1 : 0;
                if (P.invalid) P.invalid[b] = 1;
                INFO6_PUT(b, 1, (s_misc[2] == N) ? 1.0 : 0.0);
            }
        }
        __syncwarp();
    }

    // ---- job mask + candidates (always refreshed into the handle's internal buffers) ----
    {
        bool first_missing = false, unfinished = false;
        for (int j0 = 0; j0 < J; j0 += 32) {
            int j = j0 + lane;
            int nx = (j < J) ? (int)s_nxt[j] : M;
            first_missing |= __any_sync(FULL, j < J && nx == 0);
            unfinished |= __any_sync(FULL, j < J && nx < M);
        }
        double mn = INFINITY;
        for (int j = lane; j < J; j += 32) mn = fmin(mn, s_v[j]);
        mn = warp_min(mn);
        for (int j0 = 0; j0 < J; j0 += 32) {
            const int j = j0 + lane;
            uint8_t out_mask = 0;
            if (j < J) {
                int nx = s_nxt[j];
                uint8_t fin = (nx == M) ? 1 : 0;
                uint8_t esa = fin;
                if (first_missing) esa = (nx >= 1) ? 1 : 0;
                else if (unfinished) esa = (s_v[j] != mn) ? 1 : 0;
                int c = j * M + (nx < M - 1 ? nx : M - 1);
                P.jm_fin[(size_t)b * J + j] = fin;
                P.jm_esa[(size_t)b * J + j] = esa;
                P.cand_int[(size_t)b * J + j] = c;
                out_mask = (P.mask_mode == MTFJSP_MASK_ESA) ? esa : fin;
                if (MODE & MODE_OBS) {
                    if (P.jmask) P.jmask[(size_t)b * J + j] = out_mask;
                    if (P.cand) P.cand[(size_t)b * J + j] = c;
                    if (P.rec) P.rec[(size_t)b * P.rec_stride + REC_BITS + (J + 7) / 8 + j] = (uint8_t)(nx < M - 1 ? nx : M - 1);
                }
            }
            if (MODE & MODE_OBS) {
                const unsigned bits = __ballot_sync(FULL, out_mask != 0);
                if (P.rec && lane < 4 && j0 + 8 * lane < J)
                    P.rec[(size_t)b * P.rec_stride + REC_BITS + j0 / 8 + lane] = (uint8_t)(bits >> (8 * lane));
            }
        }
        if ((MODE & MODE_OBS) && P.rec)  // padding
            for (int i = REC_BITS + (J + 7) / 8 + J + lane; i < P.rec_stride; i += 32) P.rec[(size_t)b * P.rec_stride + i] = 0;
    }

    if (MODE & MODE_OBS) {
        const int rem_head = s_misc[0], fresh = s_misc[1];
        OutT* tf = reinterpret_cast<OutT*>(P.tfea);
        const double w0 = s_w[0], w1 = s_w[1], w2 = s_w[2];
        auto emit_row = [&](const int v) {
            const int mv = s_mach[v];
            const bool sch = mv >= 0, vfirst = (v % M) == 0;
            const int rp = sch ? (int)s_rpred[v] : -1;
            const bool has_job = !vfirst && v != rem_head;
            const bool co = has_job && rp == v - 1;
            const bool has_m = rp >= 0 && !co;
            if (tf) {  // SS:2246-2277
                double f[12];
                f[0] = s_st[v]; f[1] = s_ft[v]; f[2] = s_pt[v];
                f[3] = sch ? 1.0 : 0.0;
                f[4] = (double)((vfirst ? 1 : 0) + (has_job ? 1 : 0) + (has_m ? 1 : 0));
                f[5] = sch ? (double)(mv + 1) : 0.0;
                f[6] = sch ? s_dur[v] : 0.0;
                f[7] = sch ? s_psel[v] : 0.0;
                f[8] = (double)(v / M + 1);
                f[9] = w0; f[10] = w1; f[11] = w2;
                store_row<OutT>(tf + ((size_t)b * N + v) * 12, f, 12);
            }
            if (P.adj_w) {  // SS:2019-2073 in compact ELL form
                double wj = 0.0, wm = 0.0;
                int src = -1;
                if (has_job) {
                    const int u = v - 1, mu = s_mach[u];
                    double w;
                    if (fresh == v) w = s_dur[u] + s_tt[mu * M + mv] + (s_st[v] - s_ft[u]);  // SS:1764 / 1644
                    else if (s_dur[u] != 0.0) w = s_dur[u] + ((mu >= 0 && sch) ? s_tt[mu * M + mv] : 0.0);  // SS:1392-1422
                    else w = 1.0;                                                                              // SS:625,642
                    wj = adj_val(w, mu >= 0, s_dur[u]);
                }
                if (has_m) {
                    double w = s_dur[rp] + ((rp / M == v / M) ? s_tt[mv * M + mv] : 0.0) + (s_st[v] - s_ft[rp]);
                    wm = adj_val(w, true, s_dur[rp]);
                    if (wm != 0.0) src = rp;
                }
                reinterpret_cast<float2*>(P.adj_w)[(size_t)b * N + v] = make_float2((float)wj, (float)wm);
                P.adj_src[(size_t)b * N + v] = (int16_t)src;
            }
        };
        const bool inc = (MODE & MODE_STEP) && P.obs_inc;
        if (inc) {  // only the rows this step changed; an invalid action changed nothing
            if (valid) {
                for (int c = (a % M) + lane; c < M; c += 32) emit_row((a / M) * M + c);
                const int xv = lane == 0 ? o_next : lane == 1 ? rem_prev : lane == 2 ? fresh_prev : -1;
                if (xv >= 0) emit_row(xv);
            }
        } else {
            {   // route tails: last entry of each machine's range of the flat order
                int carry = 0;
                for (int m0 = 0; m0 < M; m0 += 32) {
                    const int mm = m0 + lane;
                    const int c = (mm < M) ? (int)s_cnt[mm] : 0;
                    int inc_ = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int n_ = __shfl_up_sync(FULL, inc_, o);
                        if (lane >= o) inc_ += n_;
                    }
                    if (mm < M && c > 0) s_tail[mm] = s_ord[carry + inc_ - 1];
                    carry += __shfl_sync(FULL, inc_, 31);
                }
            }
            for (int v = lane; v < N; v += 32) emit_row(v);
        }
        __syncwarp();
        if (P.mfea) {  // SS:2315-2354
            OutT* mf = reinterpret_cast<OutT*>(P.mfea);
            auto emit_mach = [&](const int mm, const int tail) {
                double f[8];
                const int c = s_cnt[mm];
                f[0] = c > 0 ? s_ft[tail] : 0.0;
                f[1] = s_macc[mm * 3 + 0]; f[2] = s_macc[mm * 3 + 1]; f[3] = s_macc[mm * 3 + 2];
                f[4] = (double)c;
                f[5] = w0; f[6] = w1; f[7] = w2;
                store_row<OutT>(mf + ((size_t)b * M + mm) * 8, f, 8);
            };
            if (inc) {
                if (valid && lane == 0) emit_mach(m, o_tail);  // the one machine row the step changed
            } else {
                for (int mm = lane; mm < M; mm += 32) emit_mach(mm, s_cnt[mm] > 0 ? (int)s_tail[mm] : 0);
            }
        }
    }
}

// =====================================================================================================
// Size-specialised kernel: (J, M) are compile-time, G lanes cooperate on one environment and a warp
// carries 32/G environments, so the scalar phases (placement decision, idle sum, reward, FP64 divisions of
// the reward scaler) are issued once for 32/G instances.  Same HBM records and arithmetic as env_kernel.
// It relies on the state invariant kept by reset and step: unscheduled ops carry their current estimate
// in st/ft (only the stepped job's chain changes per step), dur = 0 and psel = min feasible energy.
// =====================================================================================================
constexpr int calign(int x, int a) { return (x + a - 1) / a * a; }
// shape of numpy's pairwise summation of n elements (leaves of <= 128 elements, split at n/2 rounded down to a multiple
// of 8): number of leaves, longest accumulator chain of a leaf, and the combination of the leaf results
__host__ __device__ constexpr int pw_nleaf(int n) { return n <= 128 ? 1 : pw_nleaf(n / 2 - (n / 2) % 8) + pw_nleaf(n - (n / 2 - (n / 2) % 8)); }
__host__ __device__ constexpr int pw_maxchain(int n) {
    if (n <= 128) return (n - n % 8) / 8;
    const int a = pw_maxchain(n / 2 - (n / 2) % 8), b = pw_maxchain(n - (n / 2 - (n / 2) % 8));
    return a > b ? a : b;
}
template <int N_>
__device__ __forceinline__ double pw_combine(const double* leaf) {
    if constexpr (N_ <= 128) {
        return leaf[0];
    } else {
        constexpr int n2 = N_ / 2 - (N_ / 2) % 8;
        constexpr int nl = pw_nleaf(n2);
        const double x = pw_combine<n2>(leaf);
        const double y = pw_combine<N_ - n2>(leaf + nl);
        return x + y;
    }
}

// COLD_: dur / psel are not staged into shared memory (a step reads them at a handful of ops: the re-added accumulator
// chain of the energy sum and the rewritten observation rows) and the idle terms pass through a two-chunk buffer instead
// of an N-term array -- shared memory per env drops by (2N + N) doubles, which is what bounds the resident warps.
template <int J_, int M_, int G_, int WARPS_, bool COLD_ = false>
struct Spec {
    static constexpr int J = J_, M = M_, G = G_, N = J_ * M_, EPW = 32 / G_, WARPS = WARPS_;
    static constexpr bool COLD = COLD_;
    // NOTT (one env per warp, COLD): the M x M transport table is not staged either.  A step needs column m of it (lane k
    // keeps tt[k][m] in a register, read through shuffles) and a few single entries for rewritten observation rows.
    static constexpr bool NOTT = COLD_ && G_ == 32;
    static_assert(J_ <= G_ && M_ <= G_, "one lane per job and per machine");
    static constexpr int NLEAF = pw_nleaf(N), CHAIN = pw_maxchain(N);
    static_assert(N >= 8 && CHAIN <= G_, "one lane per term of an accumulator chain");
    static constexpr int NELEAF = NLEAF > 1 ? NLEAF : 0;  // a single leaf's result is the total: nothing to cache
    static constexpr int NICH = N > 128 ? (N + 31) / 32 : 0;  // cached idle-sum prefixes (one per 32 terms of the flat order)
    static_assert(NICH == 0 || G_ == 32, "idle-sum chunks are one warp wide");
    static constexpr int SD = calign(4 * N + 4 + 3 * M + 3 + 8 * NLEAF + NELEAF + NICH + 13, 2);
    static constexpr int SI = calign(3 * N + M + 3 + J, 8);
    static constexpr int XS = calign(2 * N + M * M, 2);
    static constexpr int TT = calign(M * M, 2);  // only the transport table is staged from xs
    static constexpr int O_ST = 0, O_FT = N, O_DUR = 2 * N, O_PSEL = 3 * N, O_SCAL = 4 * N, O_MACC = 4 * N + 4,
                         O_W = O_MACC + 3 * M, O_EACC = O_W + 3, O_ELEAF = O_EACC + 8 * NLEAF, O_IPRE = O_ELEAF + NELEAF,
                         O_SC = O_IPRE + NICH;
    // shared-memory image of sd: st ft [dur psel] | scal macc w eacc eleaf sc (COLD drops the bracket)
    static constexpr int HOT = COLD ? 2 * N : 4 * N, TAILBLK = SD - 4 * N, SM_SD = HOT + TAILBLK;
    static constexpr int SM_SCAL = HOT, SM_MACC = HOT + 4, SM_W = SM_MACC + 3 * M, SM_EACC = SM_W + 3,
                         SM_ELEAF = SM_EACC + 8 * NLEAF, SM_IPRE = SM_ELEAF + NELEAF, SM_SC = SM_IPRE + NICH;
    static constexpr int O_MACH = 0, O_ORD = N, O_RPRED = 2 * N, O_CNT = 3 * N, O_MISC = 3 * N + M, O_NXT = O_MISC + 3;
    static constexpr int O_MIND = 0, O_TT = 2 * N;
    // idle-term scratch: two G-term chunks (at least the three machine rows the policy mode parks there), or all N terms
    static constexpr int NPT_CHUNK = 2 * G > calign(3 * M, 4) ? 2 * G : calign(3 * M, 4), NPT_FULL = calign(N, 4);
    static constexpr int B_SD = SM_SD * 8, B_SI = SI * 2;
    static constexpr int env_bytes(int npt, int btt) {
        const int raw = calign(B_SD + btt + npt * 8 + B_SI, 16);
        // G = 8: two envs share a half-warp; offset them by 16 banks so their 8 x 8-byte rows do not collide
        return (G_ == 8) ? (raw + ((64 - raw % 128) + 128) % 128) : raw;
    }
    // blocks one SM holds by shared memory (228 KB, 1 KB reserved per block) and by threads: handed to ptxas through
    // __launch_bounds__ so that registers never become the tighter limit
    static constexpr int minb(int npt, int btt) {
        const int by_smem = 233472 / (WARPS_ * EPW * env_bytes(npt, btt) + 1024), by_threads = 2048 / (WARPS_ * 32);
        const int b = by_smem < by_threads ? by_smem : by_threads;
        return b < 32 ? b : 32;
    }
    static constexpr int B_TT = NOTT ? 0 : TT * 8;
    // CHUNK: the idle terms pass through the two-chunk buffer.  Always with COLD; without it wherever the smaller scratch
    // lets one more block onto an SM (J10M10: 18 -> 19 blocks, 3.07 -> 2.91 waves of 16,384 envs)
    static constexpr bool CHUNK = COLD_ || minb(NPT_CHUNK, B_TT) > minb(NPT_FULL, B_TT);
    static constexpr int NPT = CHUNK ? NPT_CHUNK : NPT_FULL;
    static_assert(NPT >= 3 * M, "the random-step mode parks three compacted machine rows in the idle-term scratch");
    static constexpr int B_PT = NPT * 8;
    static constexpr int RAW = calign(B_SD + B_TT + B_PT + B_SI, 16);
    static constexpr int ENV_BYTES = env_bytes(NPT, B_TT);
    static constexpr bool BAR_IN_PAD = ENV_BYTES - RAW >= 8;
    static constexpr int ITER = (N + G - 1) / G;
    static constexpr unsigned GMASK = (G_ == 32) ? 0xffffffffu : ((1u << G_) - 1u);
    static constexpr int MINB = minb(NPT, B_TT);
    // launch overlap (ovl_wait) where it was measured to pay: 4-warp blocks of 16 short envs (J6M6 random step at 65,536
    // envs, 4.6 waves: 62.5 -> 59.2 us).  The one-warp blocks of the other sizes lost with it (J10M10 at 16,384 envs
    // 34.7 -> 35.5 us, J30M20 at 4,096 envs 32.2 -> 36.6 us; profiles/README.md, round 5)
    static constexpr bool OVL = WARPS_ > 1;
};

// bulk async copy global -> shared (TMA, 1-D), completion counted in bytes on an mbarrier; 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint32_t bar) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d),
                 "l"(gmem_src), "r"(bytes), "r"(bar)
                 : "memory");
}

template <int G>
__device__ __forceinline__ double gmax_d(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
template <int G>
__device__ __forceinline__ double gmin_d(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
// 32-bit reductions over a lane group: one redux.sync with the group's member mask (the groups of a warp execute it
// together, each with its own mask) instead of log2(G) shuffle + min/max pairs
__device__ __forceinline__ unsigned gmin_u(unsigned v, unsigned gmask) { return __reduce_min_sync(gmask, v); }


// adj_val without the 64-bit integer round trip: trunc() is exact for |w| < 2^53
__device__ __forceinline__ double adj_val_t(double w, bool u_assigned, double dur_u) {
    const double wi = trunc(w);
    if (wi == 0.0) return 0.0;
    const double nd = u_assigned ? dur_u : 1.0;
    return trunc(wi - nd) + 1.0;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
// one 64-bit value per (seed, env, step): the job draw is its high half (stream 0), the machine draw its low half (stream 1)
__device__ __forceinline__ uint64_t rand_u64(uint64_t seed, uint64_t env, uint64_t step) {
    return splitmix64(seed ^ splitmix64(env * 0x100000001B3ULL + step * 0x9E3779B1ULL));
}
__device__ __forceinline__ uint32_t rand_u32(uint64_t seed, uint64_t env, uint64_t step, uint64_t stream) {
    const uint64_t x = rand_u64(seed, env, step);
    return stream == 0 ? (uint32_t)(x >> 32) : (uint32_t)x;
}

// numpy pairwise sum of up to M (<= 64) values held in registers/local array
__device__ __forceinline__ double np_sum_small(const double* a, int n) {
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    }
    double r[8];
    for (int i = 0; i < 8; i++) r[i] = a[i];
    int nb = n - (n & 7), i;
    for (i = 8; i < nb; i += 8)
        for (int k = 0; k < 8; k++) r[k] += a[i + k];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}

// position of the k-th (0-based) set bit of `bits`, -1 if there are not that many (fns.b32: n-th set bit from bit 0 up)
__device__ __forceinline__ int kth_set_bit(unsigned bits, int k, int /*maxk*/) { return (int)__fns(bits, 0u, k + 1); }

// Launch overlap (Params::done_ep).  Back-to-back whole-batch random steps of one handle are issued with programmatic
// stream serialization (launch_spec says when) and every block of a whole-batch step launch triggers its dependents when
// it starts, so launch k+1 becomes resident in the slots that the tail of launch k leaves empty instead of after the
// whole grid.  A warp of launch k+1 depends only on its own envs
// in launch k, so it waits for one completion entry per warp-sized env range -- indexed by the env range, not by
// blockIdx, so both walk directions map to the same entry -- instead of for the whole grid (griddepcontrol.wait).
// (Per warp rather than per block: the warps of a block share nothing, and no block barrier has to count warps that
// returned early.)
// No deadlock: a grid becomes resident only once every CTA of its predecessor has started, so every CTA a warp waits on
// is resident or finished; by induction over the launches, nothing waits on a CTA that cannot be scheduled.
// The wait is bounded (1 s of %globaltimer): on expiry the mapped host word is set -- the next call on the handle
// returns an error -- and the warp proceeds rather than hanging or trapping the device.
__device__ __forceinline__ void ovl_wait(const unsigned long long* flag, unsigned long long want, unsigned* err) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
    if (v >= want) return;
    uint64_t t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    unsigned ns = 32;
    do {
        __nanosleep(ns);
        if (ns < 1024) ns <<= 1;
        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (v < want && t - t0 > 1000000000ull) {
            *(volatile unsigned*)err = 1u;
            __threadfence_system();
            return;
        }
    } while (v < want);
}
// after every global write of the warp's envs (behind a __syncwarp): publish them.  max: an entry never decreases, so
// a wait for an epoch that has passed is always satisfied
__device__ __forceinline__ void ovl_release(unsigned long long* flag, unsigned long long ep) {
    asm volatile("red.release.gpu.global.max.u64 [%0], %1;" ::"l"(flag), "l"(ep) : "memory");
}

template <class S, int MODE, typename OutT>
__global__ void __launch_bounds__(S::WARPS * 32, S::MINB) env_kernel_s(const __grid_constant__ Params P) {
    constexpr int J = S::J, M = S::M, N = S::N, G = S::G, EPW = S::EPW, ITER = S::ITER;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gl = lane & (G - 1), ge = lane / G;
    const unsigned gmask = S::GMASK << (ge * G);  // member mask of this lane's group
    const int B = P.L.B;
    // reversed walk without a branch: ~blockIdx.x + gridDim.x = gridDim.x - 1 - blockIdx.x.  The branchless form keeps
    // the per-step instantiations at the register allocation (or better) they had when wb0 carried a run-time offset
    const unsigned flip = P.rev ? ~0u : 0u;
    const int blk = (int)((blockIdx.x ^ flip) + (gridDim.x & flip));
    const int wb0 = (blk * S::WARPS + warp) * EPW;
    // launch overlap (ovl_wait): the next launch may become resident as soon as every block of this one has started
    constexpr bool OVL = S::OVL && (MODE & MODE_STEP) && !(MODE & MODE_HOST);
    if (OVL && P.ep) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // only the random step without a recorded reset may start early (launch_spec): everything it reads is the handle's
    // own state, written by the handle's previous step launch
    constexpr bool WAITS = OVL && (MODE & MODE_POLICY) && !(MODE & MODE_FROM_RESET);
    if (wb0 >= B) return;
    const int b = wb0 + ge;
    const bool active = b < B;
    const int bc = active ? b : wb0;  // idle groups of the last warp shadow env wb0 and never store

    unsigned char* base = smem_raw + (size_t)(warp * EPW + ge) * S::ENV_BYTES;
    double* s_sd = reinterpret_cast<double*>(base);
    const double* __restrict__ s_tt = reinterpret_cast<const double*>(base + S::B_SD);
    double* __restrict__ s_pt = reinterpret_cast<double*>(base + S::B_SD + S::B_TT);
    int16_t* __restrict__ s_si = reinterpret_cast<int16_t*>(base + S::B_SD + S::B_TT + S::B_PT);
    // packed host-step record (P.rec): assembled in the idle-term scratch once the idle sum is done with it, then written
    // by the whole warp as one contiguous run of 8-byte words -- the buffer may be mapped host memory, where piecewise
    // stores would each become a PCIe write of their own
    // Staging: words 0..5 of the scratch = the six step-info doubles, behind them the record's bytes from `done` on.
    constexpr int RECW = rec_bytes(J) / 8, MBYTES = (J + 7) / 8;
    static_assert(6 + RECW - 5 <= S::NPT, "step info and record tail are staged in the idle-term scratch");
    unsigned char* const s_rec = reinterpret_cast<unsigned char*>(s_pt + 6) - REC_DONE;  // record byte i >= 40 at s_rec[i]
    constexpr bool REC_STAGED = (MODE & MODE_HOST) != 0;  // the host-step kernel
#define INFO6_S(k_, v_)                                                                      \
    do {                                                                                     \
        if constexpr (REC_STAGED) {                                                          \
            if (P.rec || P.info6) s_pt[(k_)] = (v_);                                         \
            if ((k_) == 1 && P.rec) {  /* the lane that knows `done` clears the tail first */ \
                for (int i_ = 0; i_ < RECW - 5; i_++) reinterpret_cast<uint64_t*>(s_pt + 6)[i_] = 0; \
                s_rec[REC_DONE] = (v_) != 0.0 ? 1 : 0;                                       \
            }                                                                                \
        } else {                                                                             \
            INFO6_PUT(b, (k_), (v_));                                                        \
        }                                                                                    \
    } while (0)

    double* g_sd = P.sd + (size_t)bc * S::SD;
    int16_t* g_si = P.si + (size_t)bc * S::SI;
    const double* g_xs = P.xs + (size_t)bc * S::XS;
    // fused episode reset: an instantiation of its own, so that the kernel of every other step carries none of it
    constexpr bool fr = (MODE & MODE_FROM_RESET) != 0;
    static_assert(!fr || (!S::COLD && (MODE & MODE_STEP)), "COLD reads dur / psel from the state record, not the snapshot");
#ifdef MTFJSP_DEBUG_BOUNDS  // debug builds: the snapshot records read here lie inside the batch
    if (fr) assert(bc < P.L.B && P.L.sd_stride == S::SD && P.L.si_stride == S::SI);
#endif
    const double* src_sd = fr ? P.sd0 + (size_t)bc * S::SD : g_sd;
    const int16_t* src_si = fr ? P.si0 + (size_t)bc * S::SI : g_si;

    int a = 0, m = 0;
    bool sel = false;  // MODE_POLICY, lane j: job j selectable
    int cj = 0;        //              lane j: candidate op of job j
    int nsel_step = 0; //              ops scheduled so far = the step counter of the random stream
    int eid = 0;       //              lane k: edge group of machine k (candidate-machine feature 5), independent of the action
    if constexpr ((MODE & MODE_POLICY) != 0) {
        if (gl < M && P.mfea1 != nullptr) eid = __ldg(P.edge_id + (size_t)bc * M + gl);
    }
    // the action is the head of a dependent chain (op -> t[op][m], mind row of its job): issue it first -- with launch
    // overlap, right behind the wait
    auto load_action = [&]() {
        if constexpr ((MODE & MODE_POLICY) != 0) {
            const uint8_t* jsrc = (P.mask_mode == MTFJSP_MASK_ESA ? P.jm_esa : P.jm_fin) + (size_t)bc * J;
            if (gl < J) {
                // the reset image (what reset_copy_kernel writes): no job masked, every job's candidate is its first op,
                // nothing scheduled
                sel = fr ? true : jsrc[gl] == 0;
                cj = fr ? gl * M : P.cand_int[(size_t)bc * J + gl];
            }
            nsel_step = fr ? 0 : g_si[S::O_MISC + 2];
        } else if (MODE & MODE_STEP) {
            if (P.act2) { const int2 am = __ldg(P.act2 + bc); a = am.x; m = am.y; }
            else { a = __ldg(P.op + bc); m = __ldg(P.mach + bc); }
        }
    };
    if constexpr (!WAITS) load_action();
    // ---- stage the records: one cp.async.bulk (TMA, 1-D) per record, three per env, issued by the group's first lane and
    // completing on the warp's mbarrier.  (16-byte cp.async copies spread over the G lanes -- 17 LDGSTS per lane at J6M6 --
    // were 5 % slower: 74.4 -> 70.5 us.)
    // the warp's mbarrier lives in the bank padding of its first env where there is one (J6M6: shared memory is exactly
    // what six blocks per SM leave), else behind the env regions
    uint64_t* s_bar = S::BAR_IN_PAD
                          ? reinterpret_cast<uint64_t*>(smem_raw + (size_t)(warp * EPW) * S::ENV_BYTES + S::RAW)
                          : reinterpret_cast<uint64_t*>(smem_raw + (size_t)S::WARPS * EPW * S::ENV_BYTES) + warp;
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(s_bar);
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar),
                     "r"((uint32_t)(EPW * (S::SM_SD * 8 + S::B_TT + S::SI * 2 + (fr ? (S::SD - (S::O_SC & ~1)) * 8 : 0))))
                     : "memory");
    }
    __syncwarp();
    if constexpr (WAITS && S::B_TT > 0) {  // static: needs nothing from the previous step
        if (gl == 0) bulk_g2s(base + S::B_SD, g_xs + S::O_TT, S::TT * 8, bar);
    }
    // launch overlap: everything below reads or writes what the previous step launch wrote for these envs.  The bulk
    // copies read it through the async proxy, the previous launch wrote it through the generic one: proxy fence.
    if constexpr (WAITS) {
        if (P.wait_ep) {
            if (lane == 0) ovl_wait(P.done_ep + wb0 / EPW, P.wait_ep, P.ovl_err);
            __syncwarp();
            if (gl == 0) asm volatile("fence.proxy.async.global;" ::: "memory");
        }
        load_action();
    }
    if (gl == 0) {
        if constexpr (S::COLD) {
            bulk_g2s(s_sd, g_sd, S::HOT * 8, bar);
            bulk_g2s(s_sd + S::HOT, g_sd + 4 * N, S::TAILBLK * 8, bar);
        } else {
            bulk_g2s(s_sd, src_sd, S::SD * 8, bar);
        }
        if constexpr (!WAITS && S::B_TT > 0) bulk_g2s(base + S::B_SD, g_xs + S::O_TT, S::TT * 8, bar);
        bulk_g2s(s_si, src_si, S::SI * 2, bar);
    }
    // fused reset: the reward-scaler block is the state's (the scaler runs across episodes), staged into the idle-term
    // scratch from the 16-byte word it starts in; the three weights are the caller's.  Both go over the staged snapshot
    // once it has landed.
    constexpr int SC0 = S::O_SC & ~1;
    static_assert(S::NPT >= S::SD - SC0, "the scaler block is staged in the idle-term scratch");
    double wv = 0.0;
    if constexpr (fr) {
        if (gl == 0) bulk_g2s(s_pt, g_sd + SC0, (S::SD - SC0) * 8, bar);
        if (gl < 3) wv = P.weights[(size_t)bc * 3 + gl];
    }
    double tr = 0.0, pr = 0.0;  // MODE_POLICY, lane k < M: t[op][k], p[op][k]
    int nsel = 1;
    if constexpr ((MODE & MODE_POLICY) != 0) {
        // uniform random selectable job, then uniform random feasible machine of its candidate op: the draws of
        // policy_kernel / oracle_policy_random (keyed by seed, global env index, step counter, stream)
        const unsigned jb = (__ballot_sync(FULL, sel) >> (ge * G)) & S::GMASK;
        nsel = __popc(jb);
        const uint64_t genv = P.env_offset + (uint64_t)bc;
        const uint64_t rnd = rand_u64(P.seed, genv, (uint64_t)nsel_step);
        const int kj = (int)(((rnd >> 32) * (uint64_t)nsel) >> 32);
        const int jl = kth_set_bit(jb, kj, J);
        a = __shfl_sync(FULL, cj, jl < 0 ? 0 : jl, G);
        if (nsel == 0) a = -1;
        const int ar = (a >= 0 && a < N) ? a : 0;
        if (gl < M) {
            tr = __ldg(P.t + ((size_t)bc * N + ar) * M + gl);
            pr = __ldg(P.p + ((size_t)bc * N + ar) * M + gl);
        }
        const unsigned fb = (__ballot_sync(FULL, gl < M && tr >= 0) >> (ge * G)) & S::GMASK;
        const int nf = __popc(fb);
        const int km = (int)(((rnd & 0xffffffffull) * (uint64_t)nf) >> 32);
        m = (nsel == 0) ? -1 : kth_set_bit(fb, km, M);
        if (active && gl == 0) { P.op_out[b] = a; P.mach_out[b] = m; }
    }
    bool valid = (MODE & MODE_STEP) && active && a >= 0 && a < N && m >= 0 && m < M;
    const int ac = valid ? a : 0, mc = valid ? m : 0;
    const int apos = ac % M, ja = ac / M;
    double d = 0.0, pa = 0.0, mind_r = 0.0;
    if constexpr ((MODE & MODE_POLICY) != 0) {
        d = __shfl_sync(FULL, tr, mc, G);   // an invalid action never uses d / pa
        pa = __shfl_sync(FULL, pr, mc, G);
        if (gl < M) mind_r = __ldg(g_xs + S::O_MIND + ja * M + gl);
    } else if (MODE & MODE_STEP) {
        d = __ldg(P.t + ((size_t)bc * N + ac) * M + mc);
        pa = __ldg(P.p + ((size_t)bc * N + ac) * M + mc);
        if (gl < M) mind_r = __ldg(g_xs + S::O_MIND + ja * M + gl);  // lane c: min duration of op (ja, c)
    }
    double ttcol = 0.0;  // NOTT, lane k < M: tt[k][m]
    if constexpr (S::NOTT && (MODE & MODE_STEP) != 0) {
        if (gl < M) ttcol = __ldg(g_xs + S::O_TT + gl * M + mc);
    }
    if constexpr (S::COLD && (MODE & MODE_STEP) != 0) {
        // the few dur / psel words this step reads from HBM, requested now (the action is known) so that they are in L1
        // when the energy chain and the observation rows get to them: accumulator chain and tail of the op's leaf, the
        // rows of the stepped job
        int lf = 0, loff = 0, ln = N;
        if constexpr (S::NLEAF > 1) {
#pragma unroll
            for (int q = 1; q < S::NLEAF; q++)
                if (ac >= P.pw.leaf_off[q]) lf = q;
            loff = P.pw.leaf_off[lf];
            ln = P.pw.leaf_len[lf];
        }
        const int nb = ln - (ln & 7), x = ac - loff;
        int v1 = -1;
        if (x < nb && gl < (nb >> 3)) v1 = loff + (x & 7) + 8 * gl;
        else if (gl >= 16 && gl - 16 < (ln & 7)) v1 = loff + nb + gl - 16;
        if (v1 >= 0) {
            asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_DUR + v1));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_PSEL + v1));
        }
        if (gl < M && (MODE & MODE_OBS)) {
            asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_PSEL + ja * M + gl));
            if (gl == 0 && apos > 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_DUR + ac - 1));
        }
    }
    {
        uint32_t ok;
        do {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(ok)
                : "r"(bar)
                : "memory");
        } while (!ok);
    }
    if constexpr (fr) {  // R[0..3] are the running returns a folded-in scaler reset clears
        const double* s_sc0 = s_pt + (S::O_SC - SC0);
        for (int i = gl; i < 13; i += G) s_sd[S::SM_SC + i] = (i < 4 && P.clear_ret) ? 0.0 : s_sc0[i];
        if (gl < 3) s_sd[S::SM_W + gl] = wv;
    }
    __syncwarp();

    double* __restrict__ s_st = s_sd + S::O_ST;
    double* __restrict__ s_ft = s_sd + S::O_FT;
    double* __restrict__ s_scal = s_sd + S::SM_SCAL;
    double* __restrict__ s_macc = s_sd + S::SM_MACC;
    const double* __restrict__ s_w = s_sd + S::SM_W;
    double* __restrict__ s_sc = s_sd + S::SM_SC;
    // duration / selected power of op v: shared memory, or (COLD) straight from the state record in HBM.  The stepped
    // op's own values are in registers (d, pa): its HBM words are written by this very launch.
    auto TT = [&](const int i, const int j) -> double {
        if constexpr (S::NOTT) return __ldg(g_xs + S::O_TT + i * M + j);
        else return s_tt[i * M + j];
    };
    bool stepped = false;  // set once the action is known to be valid
    auto DUR = [&](const int v) -> double {
        if constexpr (S::COLD) return (stepped && v == ac) ? d : g_sd[S::O_DUR + v];
        else return s_sd[S::O_DUR + v];
    };
    auto PSEL = [&](const int v) -> double {
        if constexpr (S::COLD) return (stepped && v == ac) ? pa : g_sd[S::O_PSEL + v];
        else return s_sd[S::O_PSEL + v];
    };
    int16_t* __restrict__ s_mach = s_si + S::O_MACH;
    int16_t* __restrict__ s_ord = s_si + S::O_ORD;
    int16_t* __restrict__ s_rpred = s_si + S::O_RPRED;
    int16_t* __restrict__ s_cnt = s_si + S::O_CNT;
    int16_t* __restrict__ s_misc = s_si + S::O_MISC;
    int16_t* __restrict__ s_nxt = s_si + S::O_NXT;

    // NOTT: feature 2 of the candidate-machine row is a transport-table entry that comes straight from HBM; its pair is
    // stored after the placement scan so that the load's latency is not waited for here
    double mf_f2 = 0.0, mf_f3 = 0.0;
    bool mf_pending = false;
    if constexpr ((MODE & MODE_POLICY) != 0) {
        // candidate-machine features of the drawn op (trainer/parallel_env.py:152-214), lane k = machine k; the means
        // run over the positive entries in machine order = numpy's sum of the compacted row (np_sum_small)
        if (P.mfea1 != nullptr) {
            const double ptl = tr * fabs(pr);
            const bool qt = gl < M && tr > 0, qpt = gl < M && ptl > 0, qp = gl < M && pr > 0;
            const unsigned bt = (__ballot_sync(FULL, qt) >> (ge * G)) & S::GMASK;
            const unsigned bpt = (__ballot_sync(FULL, qpt) >> (ge * G)) & S::GMASK;
            const unsigned bp = (__ballot_sync(FULL, qp) >> (ge * G)) & S::GMASK;
            const unsigned lt = (1u << gl) - 1u;
            if (qt) s_pt[__popc(bt & lt)] = tr;
            if (qpt) s_pt[M + __popc(bpt & lt)] = ptl;
            if (qp) s_pt[2 * M + __popc(bp & lt)] = pr;
            __syncwarp();
            const int which = gl % 3;  // lanes 0, 1, 2 of the group: mean t, mean t*|p|, mean p (one division each)
            const int cnt = which == 0 ? __popc(bt) : which == 1 ? __popc(bpt) : __popc(bp);
            const double mean_w = np_sum_small(s_pt + which * M, cnt) / (double)cnt;
            const double mean_t = __shfl_sync(FULL, mean_w, 0, G);
            const double mean_pt = __shfl_sync(FULL, mean_w, 1, G);
            const double mean_p = __shfl_sync(FULL, mean_w, 2, G);
            if (active && nsel > 0 && gl < M) {
                int pm_row = M - 1;  // int(tfea[a-1][5]) - 1 wraps to the last row while the predecessor is unscheduled
                if (a % M != 0) {
                    const int mp = s_mach[a - 1];
                    if (mp >= 0) pm_row = mp;
                }
                const int infeasible = !(tr >= 0);
                const double f0 = tr > 0 ? tr : mean_t, f1 = ptl > 0 ? ptl : mean_pt;
                const double f2 = (a % M == 0) ? 0.0 : TT(pm_row, gl);
                const double f3 = (double)(1 - infeasible), f4 = pr > 0 ? pr : mean_p;
                const double f5 = (double)eid;
                OutT* o = reinterpret_cast<OutT*>(P.mfea1) + ((size_t)b * M + gl) * 6;
                if constexpr (sizeof(OutT) == 4) {
                    float2* o2 = reinterpret_cast<float2*>(o);
                    o2[0] = make_float2((float)f0, (float)f1);
                    if constexpr (!S::NOTT) o2[1] = make_float2((float)f2, (float)f3);
                    o2[2] = make_float2((float)f4, (float)f5);
                } else {
                    double2* o2 = reinterpret_cast<double2*>(o);
                    o2[0] = make_double2(f0, f1);
                    if constexpr (!S::NOTT) o2[1] = make_double2(f2, f3);
                    o2[2] = make_double2(f4, f5);
                }
                if constexpr (S::NOTT) { mf_f2 = f2; mf_f3 = f3; mf_pending = true; }
                if (P.mmask) P.mmask[(size_t)b * M + gl] = (uint8_t)infeasible;
            }
            __syncwarp();  // s_pt is reused by the idle terms
        }
    }

    bool done = false;
    double idle = 0.0, nt = 0.0, trans = 0.0, ec = 0.0;
    // for the incremental observation: the op that now follows the stepped op on its machine, the machine's last op,
    // and the one-step transients (removed job arc, coincident arc) of the PREVIOUS step, whose rows revert now
    int o_next = -1, o_tail = -1, rem_prev = -1, fresh_prev = -1;

    if (MODE & MODE_STEP) {
        const int nsched0 = s_misc[2];
        rem_prev = s_misc[0];
        fresh_prev = s_misc[1];
        const bool first = apos == 0;
        const int aprev = first ? ac : ac - 1;
        valid = valid && nsched0 < N && (s_mach[ac] < 0) && (first || s_mach[aprev] >= 0) && !(d < 0);
        stepped = valid;
        int mp = s_mach[aprev];
        mp = (first || mp < 0) ? 0 : mp;
        double tt_pa, ttmm;  // tt[machine of the job predecessor][m], tt[m][m]
        if constexpr (S::NOTT) {
            tt_pa = __shfl_sync(FULL, ttcol, mp);
            ttmm = __shfl_sync(FULL, ttcol, mc);
        } else {
            tt_pa = TT(mp, mc);
            ttmm = TT(mc, mc);
        }
        const double arr_a = first ? 0.0 : s_ft[aprev] + tt_pa;  // DGenv_func.py:46-66
        const int len = s_cnt[mc];
        const double lbft = arr_a + d;
        // machine k's route is ord[off_k, off_k + cnt[k]): exclusive scan of the route lengths over the group's lanes
        int offm;
        {
            const int c = (gl < M) ? (int)s_cnt[gl] : 0;
            int inc = c;
#pragma unroll
            for (int o = 1; o < G; o <<= 1) {
                const int n_ = __shfl_up_sync(FULL, inc, o, G);
                if (gl >= o) inc += n_;
            }
            offm = __shfl_sync(FULL, inc - c, mc, G);
        }
        // one pass over the route of machine m (not over all ops): first feasible slot, SS:1548-1601
        unsigned best = 0xffffffffu;
        const int lastop = len > 0 ? (int)s_ord[offm + len - 1] : -1;
        if (P.L.left_shift) {
            // NOTT: tt[.][m] comes from a shuffle, so every lane walks ceil(len / G) chunks (one env per warp: uniform)
            const int kend = S::NOTT ? ((len + G - 1) / G) * G : len;
            for (int k = gl; k < kend; k += G) {
                const bool in = k < len;
                const int v = in ? (int)s_ord[offm + k] : 0;
                const bool vfirst = (v % M) == 0;
                const int vp = vfirst ? v : v - 1;
                int mvp = s_mach[vp];
                mvp = mvp < 0 ? 0 : mvp;
                double ttv;
                if constexpr (S::NOTT) ttv = __shfl_sync(FULL, ttcol, mvp);
                else ttv = TT(mvp, mc);
                if (in) {
                    double nst = vfirst ? 0.0 : s_ft[vp] + ttv;
                    bool ok;
                    if (k == 0) {
                        ok = (lbft <= nst);  // SS:1548
                    } else {
                        const int rp = s_ord[offm + k - 1];
                        const double val = s_ft[rp] + ((rp / M == v / M) ? ttmm : 0.0);
                        nst = fmax(nst, val);
                        ok = !(lbft > nst) && !((nst - s_ft[rp]) < d);  // SS:1597-1601
                    }
                    if (ok) best = min(best, ((unsigned)k << 16) | (unsigned)v);
                }
            }
        }
        best = gmin_u(best, gmask);
        if constexpr (S::NOTT && (MODE & MODE_POLICY) != 0) {
            if (mf_pending) {
                OutT* o = reinterpret_cast<OutT*>(P.mfea1) + ((size_t)b * M + gl) * 6;
                if constexpr (sizeof(OutT) == 4) reinterpret_cast<float2*>(o)[1] = make_float2((float)mf_f2, (float)mf_f3);
                else reinterpret_cast<double2*>(o)[1] = make_double2(mf_f2, mf_f3);
            }
        }
        double st = arr_a;
        int where = 0, prev = -1, next = -1, rem_head = -1, fresh = -1;
        if (len > 0) {
            if (best != 0xffffffffu) {
                where = (int)(best >> 16);
                next = (int)(best & 0xffffu);
                if (where > 0) {
                    prev = s_rpred[next];
                    const double y = s_ft[prev] + ((prev / M == ja) ? ttmm : 0.0);  // SS:1619
                    st = (y > arr_a) ? y : arr_a;
                    if (next == prev + 1 && (next % M) != 0) rem_head = next;  // SS:1660
                }
            } else {  // _append_at_the_end, SS:1689-1775
                where = len;
                prev = lastop < 0 ? 0 : lastop;
                const double y = s_ft[prev] + ((prev / M == ja) ? ttmm : 0.0);
                st = (y > arr_a) ? y : arr_a;
            }
            if (prev >= 0 && prev == ac - 1 && !first) fresh = ac;
        }
        o_next = next;
        o_tail = (where == len || lastop < 0) ? ac : lastop;
        if constexpr (S::COLD && (MODE & MODE_OBS) != 0) {  // rows of the follower and of last step's transients: dur / psel
            const int pv = gl == 0 ? next : gl == 1 ? rem_prev : gl == 2 ? fresh_prev : gl == 3 ? next - 1 : gl == 4 ? rem_prev - 1
                                                                                                  : gl == 5 ? fresh_prev - 1 : -1;
            if (pv >= 0) {
                asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_DUR + pv));
                if (gl < 3) asm volatile("prefetch.global.L1 [%0];" ::"l"(g_sd + S::O_PSEL + pv));
            }
        }
        // estimator chain of the job's remaining ops (SS:1964-1995): lane c ends up with op (ja, c)
        double my_st = 0.0, my_ft = 0.0;
        {
            double cur = st + d;
#pragma unroll
            for (int c = 1; c < M; c++) {
                const double mdc = __shfl_sync(FULL, mind_r, c, G);
                if (c > apos) {
                    const double s0 = cur;
                    cur = cur + mdc;
                    if (gl == c) { my_st = s0; my_ft = cur; }
                }
            }
        }
        __syncwarp();
        // ---- apply: open slot p of the flat order (entries behind it move up by one, highest chunk first) ----
        const int p = offm + where;
        {
            const int it_lo = (G == 32) ? (p / G) : 0;  // one env per warp: the trip count is warp-uniform
#pragma unroll
            for (int it = ITER - 1; it >= 0; --it) {
                if (it < it_lo) break;
                const int g = gl + it * G;
                const bool mv_ = valid && g >= p && g < nsched0;
                const int16_t x = mv_ ? s_ord[g] : (int16_t)0;
                __syncwarp();
                if (mv_) { s_ord[g + 1] = x; g_si[S::O_ORD + g + 1] = x; }
            }
        }
        if (valid && gl > apos && gl < M) {
            const int idx = ja * M + gl;
            s_st[idx] = my_st; s_ft[idx] = my_ft;
            g_sd[S::O_ST + idx] = my_st; g_sd[S::O_FT + idx] = my_ft;
        }
        __syncwarp();
        if (valid && gl == 0) {
            s_mach[ac] = (int16_t)mc; s_ord[p] = (int16_t)ac; s_rpred[ac] = (int16_t)prev;
            if (next >= 0) s_rpred[next] = (int16_t)ac;
            s_cnt[mc] = (int16_t)(len + 1);
            s_misc[0] = (int16_t)rem_head; s_misc[1] = (int16_t)fresh; s_misc[2] = (int16_t)(nsched0 + 1);
            s_nxt[ja] = (int16_t)(apos + 1);
            s_st[ac] = st; s_ft[ac] = st + d;
            if constexpr (!S::COLD) { s_sd[S::O_DUR + ac] = d; s_sd[S::O_PSEL + ac] = pa; }
            g_si[S::O_MACH + ac] = (int16_t)mc; g_si[S::O_ORD + p] = (int16_t)ac; g_si[S::O_RPRED + ac] = (int16_t)prev;
            if (next >= 0) g_si[S::O_RPRED + next] = (int16_t)ac;
            g_si[S::O_CNT + mc] = (int16_t)(len + 1);
            g_si[S::O_MISC + 0] = (int16_t)rem_head; g_si[S::O_MISC + 1] = (int16_t)fresh;
            g_si[S::O_MISC + 2] = (int16_t)(nsched0 + 1);
            g_si[S::O_NXT + ja] = (int16_t)(apos + 1);
            g_sd[S::O_ST + ac] = st; g_sd[S::O_FT + ac] = st + d; g_sd[S::O_DUR + ac] = d; g_sd[S::O_PSEL + ac] = pa;
        }
        __syncwarp();
        const int nsched = nsched0 + (valid ? 1 : 0);
        done = (nsched == N);
        // ---- idle time: sequential sum in (machine, route) order, DGenv_func.py:144-170 ----
        if constexpr (S::CHUNK) {
            // terms in (machine, route) order = flat order, G at a time through a two-chunk buffer: chunk i is summed
            // (a chain of dependent additions in the reference's order, on every lane) while chunk i + 1 is being written
            const int nchunk = (__reduce_max_sync(FULL, nsched) + G - 1) / G;
            // the terms in front of the chunk the op went into are the previous step's: restart from the cached running
            // sum there (terms behind the slot moved up by one, the follower's changed) and refresh the cache on the way
            int c0 = 0;
            if constexpr (S::NICH > 0) {
                c0 = valid ? (p >> 5) : 0;
                idle = s_sd[S::SM_IPRE + c0];
            }
            for (int it = c0; it < nchunk; it++) {
                if constexpr (S::NICH > 0) {
                    if (valid && it > c0 && gl == 0) { s_sd[S::SM_IPRE + it] = idle; g_sd[S::O_IPRE + it] = idle; }
                }
                const int g = gl + it * G;
                double term = 0.0;   // x + 0.0 == x exactly (gaps are never -0.0): slots past the env's term count add nothing
                if (g < nsched) {
                    const int v = s_ord[g], rp = s_rpred[v];
                    term = (rp < 0) ? (s_st[v] - 0.0) : (s_st[v] - s_ft[rp]);
                }
                double* buf = s_pt + (it & 1) * G;
                buf[gl] = term * 1.0;
                __syncwarp();
                const double2* t2 = reinterpret_cast<const double2*>(buf);
#pragma unroll
                for (int q = 0; q < G / 2; q += 2) {
                    const double2 ta = t2[q], tb = t2[q + 1];
                    idle = idle + ta.x;
                    idle = idle + ta.y;
                    idle = idle + tb.x;
                    idle = idle + tb.y;
                }
            }
            if constexpr (S::NICH > 0) {  // a full last chunk: the next op may open chunk `nchunk`
                if (valid && gl == 0 && nchunk * G == nsched && nchunk < S::NICH && nchunk > c0) {
                    s_sd[S::SM_IPRE + nchunk] = idle; g_sd[S::O_IPRE + nchunk] = idle;
                }
            }
        } else {
            // terms in (machine, route) order = flat order; a route head's term is its start time
#pragma unroll
            for (int it = 0; it < ITER; it++) {
                const int g = gl + it * G;
                if (g < nsched) {
                    const int v = s_ord[g], rp = s_rpred[v];
                    const double term = (rp < 0) ? (s_st[v] - 0.0) : (s_st[v] - s_ft[rp]);
                    s_pt[g] = term * 1.0;
                }
            }
            // the sum is a chain of dependent additions in the reference's order; x + 0.0 == x exactly (gaps are never
            // -0.0), so the slots between this env's term count and the warp's trip count are zero-filled and the loop
            // needs no per-term predicates: two 16-byte loads and four additions per four terms
            const int nmax4 = (__reduce_max_sync(FULL, nsched) + 3) & ~3;
            static_assert(S::CHUNK || S::B_PT >= ((N + 3) & ~3) * 8, "the padded idle sum reads whole groups of four terms");
            for (int g = nsched + gl; g < nmax4; g += G) s_pt[g] = 0.0;
            __syncwarp();
            const double2* t2 = reinterpret_cast<const double2*>(s_pt);
            for (int g = 0; g < nmax4; g += 4) {
                const double2 ta = t2[g >> 1], tb = t2[(g >> 1) + 1];
                idle = idle + ta.x;
                idle = idle + ta.y;
                idle = idle + tb.x;
                idle = idle + tb.y;
            }
        }
        nt = first ? 0.0 : tt_pa;  // SS:872-877
        trans = s_scal[2] + nt;
        ec = pa * d;
        __syncwarp();
    }

    // per job (lane j): ops scheduled so far, ESA key = finish of its last scheduled op, row maximum
    int nx = 0;
    double vj = INFINITY, jmx = -INFINITY;
    if (gl < J) {
        nx = s_nxt[gl];
        const double lastft = s_ft[gl * M + (nx > 0 ? nx - 1 : 0)];
        vj = (nx == M) ? INFINITY : (nx > 0 ? lastft : 0.0);
        jmx = s_ft[gl * M + M - 1];  // times are non-decreasing along a job (t >= 0, tt >= 0)
    }
    __syncwarp();

    if (MODE & MODE_STEP) {
        const double mkv = gmax_d<G>(jmx);  // SS:894
        // ---- energy estimate (SS:896): np.sum over all ops of (scheduled ? t * p : min energy), numpy's pairwise
        // summation.  Only the stepped op's term changed, so of the cached per-leaf state (8 accumulators r[k] = a[k] +
        // a[8+k] + ..., then ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail elements one by one) only accumulator
        // (x mod 8) of the op's leaf is re-added -- every addition in numpy's order, so the total is bit-identical to
        // a full recomputation (which the generic kernel does, and the parity suite compares).
        double en;
        {
            double* __restrict__ s_eacc = s_sd + S::SM_EACC;
            double* __restrict__ s_eleaf = s_sd + S::SM_ELEAF;
            int lf = 0, loff = 0, ln = N;
            if constexpr (S::NLEAF > 1) {
#pragma unroll
                for (int q = 1; q < S::NLEAF; q++)
                    if (ac >= P.pw.leaf_off[q]) lf = q;
                loff = P.pw.leaf_off[lf];
                ln = P.pw.leaf_len[lf];
            }
            const int nb = ln - (ln & 7), x = ac - loff, k = x & 7;
            constexpr int TAILMAX = S::NLEAF > 1 ? 7 : (N & 7);  // a single leaf: the tail length is known at compile time
            auto ept_of = [&](const int v) { return (s_mach[v] >= 0) ? DUR(v) * PSEL(v) : PSEL(v); };
            // accumulator chain k: lane i fetches term i, the additions run in order on every lane of the group
            const int nterm = (x < nb) ? (nb >> 3) : 0;
            const double term = (gl < nterm) ? ept_of(loff + k + 8 * gl) : 0.0;
            double r = __shfl_sync(FULL, term, 0, G);
#pragma unroll
            for (int i = 1; i < S::CHAIN; i++) {
                const double t_ = __shfl_sync(FULL, term, i, G);
                if (i < nterm) r = r + t_;
            }
            if (valid && nterm > 0 && gl == 0) { s_eacc[lf * 8 + k] = r; g_sd[S::O_EACC + lf * 8 + k] = r; }
            __syncwarp();
            double e8 = s_eacc[lf * 8 + (gl & 7)];
            e8 = e8 + __shfl_down_sync(FULL, e8, 1, 8);
            e8 = e8 + __shfl_down_sync(FULL, e8, 2, 8);
            e8 = e8 + __shfl_down_sync(FULL, e8, 4, 8);
            double leaf = __shfl_sync(FULL, e8, 0, G);
            const int ntail = ln & 7;
            const double tl = (gl < ntail) ? ept_of(loff + nb + gl) : 0.0;
#pragma unroll
            for (int i = 0; i < TAILMAX; i++) {
                const double t_ = __shfl_sync(FULL, tl, i, G);
                if (i < ntail) leaf = leaf + t_;
            }
            if constexpr (S::NLEAF > 1) {
                if (valid && gl == 0) { s_eleaf[lf] = leaf; g_sd[S::O_ELEAF + lf] = leaf; }
                __syncwarp();
                en = pw_combine<N>(s_eleaf);
            } else {
                en = leaf;
            }
        }
        // ---- reward (SS:1066-1132) and reward scaling (ppo_trick.py:73-88,115-119) ----
        const double mk_prev = s_scal[0], e_prev = s_scal[1], trans_prev = s_scal[2], idle_prev = s_scal[3];
        const double q = ((gl & 1) ? ec : (1.0 * e_prev - en)) / (double)N;  // one division sequence for both
        const double r_pt = __shfl_sync(FULL, q, 0, G);
        const double ecn = __shfl_sync(FULL, q, 1, G);
        const double r_t = 1.0 * mk_prev - mkv;
        const double r_tt = 1.0 * trans_prev - trans;
        const double r_idle = 1.0 * idle_prev - idle;
        double total = P.cfgw[0] * r_t + P.cfgw[1] * (r_pt + 1.0 * r_idle) + P.cfgw[2] * r_tt * 1.0;
        if (P.divisor != 1.0) total = total / P.divisor;
        const int k4 = gl & 3;
        const double x = k4 == 0 ? r_t : k4 == 1 ? r_idle : k4 == 2 ? r_pt : r_tt;  // parallel_env.py:255
        const double R = P.gamma * s_sc[k4] + x;
        const double nn = s_sc[12] + 1.0;
        const double old = s_sc[4 + k4], S0 = s_sc[8 + k4];
        const double mean1 = old + (R - old) / nn;
        const double S1 = S0 + (R - old) * (R - mean1);
        const double sd1 = sqrt(S1 / nn);
        const bool firstn = (nn == 1.0);
        const double mean = firstn ? R : mean1, Sn = firstn ? S0 : S1, sdv = firstn ? fabs(R) : sd1;
        const double scaled = x / (sdv + 1e-8);
        __syncwarp();
        if (valid) {
            if (gl < 4) {
                s_sc[gl] = R; s_sc[4 + gl] = mean; s_sc[8 + gl] = Sn;
                if (P.scaled4) P.scaled4[(size_t)b * 4 + gl] = scaled;
                INFO6_S(2 + gl, scaled);
            }
            if (gl == 0) {
                s_sc[12] = nn;
                s_macc[mc * 3 + 0] += ecn;  // SS:2323-2338
                s_macc[mc * 3 + 1] += nt;
                s_macc[mc * 3 + 2] += idle - idle_prev;
                s_scal[0] = mkv; s_scal[1] = en; s_scal[2] = trans; s_scal[3] = idle;  // SS:932-936
                if (P.reward5) {
                    double* r5 = P.reward5 + (size_t)b * 5;
                    r5[0] = total; r5[1] = r_t; r5[2] = r_idle; r5[3] = r_pt; r5[4] = r_tt;
                }
                if (P.done) P.done[b] = done ? 1 : 0;
                if (P.invalid) P.invalid[b] = 0;
                INFO6_S(0, total); INFO6_S(1, done ? 1.0 : 0.0);
            }
        } else if (active) {
            if (gl < 5 && P.reward5) P.reward5[(size_t)b * 5 + gl] = 0.0;
            if (gl < 4 && P.scaled4) P.scaled4[(size_t)b * 4 + gl] = 0.0;
            if (gl < 6 && gl != 1) INFO6_S(gl, 0.0);
            if (gl == 0) {
                if (P.done) P.done[b] = (s_misc[2] == N) ? 1 : 0;
                if (P.invalid) P.invalid[b] = 1;
                INFO6_S(1, (s_misc[2] == N) ? 1.0 : 0.0);
            }
        }
        __syncwarp();
        if (valid && !fr) {  // selective write-back: 4 scalars, macc[m][3], 13 scaler words
#pragma unroll
            for (int i = gl; i < 20; i += G) {
                if (i < 4) g_sd[S::O_SCAL + i] = s_scal[i];
                else if (i < 7) g_sd[S::O_MACC + mc * 3 + (i - 4)] = s_macc[mc * 3 + (i - 4)];
                else g_sd[S::O_SC + (i - 7)] = s_sc[i - 7];
            }
        }
    }

    // ---- job mask + candidates (ppo_algorithm.py:202-317) ----
    {
        const unsigned bal0 = __ballot_sync(FULL, gl < J && nx == 0);
        const unsigned bal1 = __ballot_sync(FULL, gl < J && nx < M);
        const bool first_missing = ((bal0 >> (ge * G)) & S::GMASK) != 0;
        const bool unfinished = ((bal1 >> (ge * G)) & S::GMASK) != 0;
        const double mn = gmin_d<G>(vj);
        uint8_t out_mask = 0;
        if (gl < J && active) {
            const uint8_t fin = (nx == M) ? 1 : 0;
            uint8_t esa = fin;
            if (first_missing) esa = (nx >= 1) ? 1 : 0;
            else if (unfinished) esa = (vj != mn) ? 1 : 0;
            const int c = gl * M + (nx < M - 1 ? nx : M - 1);
            P.jm_fin[(size_t)b * J + gl] = fin;
            P.jm_esa[(size_t)b * J + gl] = esa;
            P.cand_int[(size_t)b * J + gl] = c;
            out_mask = (P.mask_mode == MTFJSP_MASK_ESA) ? esa : fin;
            if (MODE & MODE_OBS) {
                if (P.jmask) P.jmask[(size_t)b * J + gl] = out_mask;
                if (P.cand) P.cand[(size_t)b * J + gl] = c;
            }
        }
        if ((MODE & MODE_OBS) && P.rec) {  // mask bits and next-op bytes of the packed record
            const unsigned bits = (__ballot_sync(FULL, out_mask != 0) >> (ge * G)) & S::GMASK;
            unsigned char* const r = REC_STAGED ? s_rec : P.rec + (size_t)b * P.rec_stride;
            if (active) {
                if (gl < MBYTES) r[REC_BITS + gl] = (uint8_t)(bits >> (8 * gl));
                if (gl < J) r[REC_BITS + MBYTES + gl] = (uint8_t)(nx < M - 1 ? nx : M - 1);
                if (!REC_STAGED)
                    for (int i = REC_BITS + MBYTES + J + gl; i < RECW * 8; i += G) r[i] = 0;
            }
        }
        if constexpr (REC_STAGED) {
            const unsigned char* const wbase = smem_raw + (size_t)(warp * EPW) * S::ENV_BYTES + S::B_SD + S::B_TT;
            if (P.rec || P.info6) __syncwarp();
            if (P.info6) {  // [B,6] step info: the warp's EPW rows are contiguous, 16 bytes per lane
                double2* const out = reinterpret_cast<double2*>(P.info6 + (size_t)wb0 * 6);
#pragma unroll
                for (int i0 = 0; i0 < EPW * 3; i0 += 32) {
                    const int i = i0 + lane, e = i / 3, w = i - e * 3;
                    if (i < EPW * 3 && wb0 + e < B)
                        out[i] = *reinterpret_cast<const double2*>(wbase + (size_t)e * S::ENV_BYTES + w * 16);
                }
            }
            if (P.rec) {  // the warp's EPW records are contiguous in the output
                auto word = [&](const int i) {  // 8-byte word i of the warp's run: r | scaled[4] | tail words
                    const int e = i / RECW, w = i - e * RECW;
                    return *reinterpret_cast<const double*>(wbase + (size_t)e * S::ENV_BYTES + (w == 0 ? 0 : w + 1) * 8);
                };
                if constexpr ((EPW * RECW) % 2 == 0) {
                    // 16 bytes per lane: over PCIe 47.5 GB/s against 43.7 with 8-byte lanes (profiles/micro/hostwrite.cu)
                    double2* const out = reinterpret_cast<double2*>(P.rec + (size_t)wb0 * (RECW * 8));
#pragma unroll
                    for (int i0 = 0; i0 < EPW * RECW / 2; i0 += 32) {
                        const int i = i0 + lane;
                        if (i < EPW * RECW / 2 && wb0 + (2 * i + 1) / RECW < B) out[i] = make_double2(word(2 * i), word(2 * i + 1));
                        else if (i < EPW * RECW / 2 && wb0 + (2 * i) / RECW < B) reinterpret_cast<double*>(out)[2 * i] = word(2 * i);
                    }
                } else {
                    double* const out = reinterpret_cast<double*>(P.rec + (size_t)wb0 * (RECW * 8));
#pragma unroll
                    for (int i0 = 0; i0 < EPW * RECW; i0 += 32) {
                        const int i = i0 + lane;
                        if (i < EPW * RECW && wb0 + i / RECW < B) out[i] = word(i);
                    }
                }
            }
        }
    }

    if (MODE & MODE_OBS) {
        const int rem_head = s_misc[0], fresh = s_misc[1];
        OutT* tf = reinterpret_cast<OutT*>(P.tfea);
        const OutT w0 = (OutT)s_w[0], w1 = (OutT)s_w[1], w2 = (OutT)s_w[2];
        // feature row (SS:2246-2277) and compact ELL adjacency row (SS:2019-2073) of op v; eptv = its estimated energy
        auto emit_row = [&](const int v, const double eptv) {
            const int mv = s_mach[v];
            const bool sch = mv >= 0, vfirst = (v % M) == 0;
            const int rp = sch ? (int)s_rpred[v] : -1;
            const bool has_job = !vfirst && v != rem_head;
            const bool co = has_job && rp == v - 1;
            const bool has_m = rp >= 0 && !co;
            const double stv = s_st[v], ftv = s_ft[v], durv = DUR(v);
            if (tf) {
                const int indeg = (vfirst ? 1 : 0) + (has_job ? 1 : 0) + (has_m ? 1 : 0);
                OutT* row = tf + ((size_t)b * N + v) * 12;
                if constexpr (sizeof(OutT) == 4) {
                    float4* r4 = reinterpret_cast<float4*>(row);
                    r4[0] = make_float4((float)stv, (float)ftv, (float)eptv, sch ? 1.f : 0.f);
                    r4[1] = make_float4((float)indeg, (float)(mv + 1), (float)durv, sch ? (float)PSEL(v) : 0.f);
                    r4[2] = make_float4((float)(v / M + 1), w0, w1, w2);
                } else {
                    double2* r2 = reinterpret_cast<double2*>(row);
                    r2[0] = make_double2(stv, ftv);
                    r2[1] = make_double2(eptv, sch ? 1.0 : 0.0);
                    r2[2] = make_double2((double)indeg, (double)(mv + 1));
                    r2[3] = make_double2(durv, sch ? PSEL(v) : 0.0);
                    r2[4] = make_double2((double)(v / M + 1), w0);
                    r2[5] = make_double2(w1, w2);
                }
            }
            if (P.adj_w) {
                double wj = 0.0, wm = 0.0;
                int src = -1;
                if (has_job) {
                    const int u = v - 1, mu = s_mach[u];
                    const double du = DUR(u);
                    double w;
                    if (fresh == v) w = du + TT(mu, mv) + (stv - s_ft[u]);                 // SS:1764 / 1644
                    else if (du != 0.0) w = du + ((mu >= 0 && sch) ? TT(mu, mv) : 0.0);   // SS:1392-1422
                    else w = 1.0;                                                                  // SS:625,642
                    wj = adj_val_t(w, mu >= 0, du);
                }
                if (has_m) {
                    const double dr = DUR(rp);
                    const double w = dr + ((rp / M == v / M) ? TT(mv, mv) : 0.0) + (stv - s_ft[rp]);
                    wm = adj_val_t(w, true, dr);
                    if (wm != 0.0) src = rp;
                }
                reinterpret_cast<float2*>(P.adj_w)[(size_t)b * N + v] = make_float2((float)wj, (float)wm);
                P.adj_src[(size_t)b * N + v] = (int16_t)src;
            }
        };
        // machine feature row k (SS:2315-2354); tail = last op of its route
        auto emit_mach = [&](const int k, const int tail) {
            OutT* mf = reinterpret_cast<OutT*>(P.mfea);
            double f[8];
            const int c = s_cnt[k];
            f[0] = c > 0 ? s_ft[tail] : 0.0;
            f[1] = s_macc[k * 3 + 0]; f[2] = s_macc[k * 3 + 1]; f[3] = s_macc[k * 3 + 2];
            f[4] = (double)c;
            f[5] = s_w[0]; f[6] = s_w[1]; f[7] = s_w[2];
            store_row<OutT>(mf + ((size_t)b * M + k) * 8, f, 8);
        };
        // Incremental observation (P.obs_inc): the output buffers hold the observation of the previous step.  A step
        // changes the rows of the stepped job from the stepped op on (its start / finish / machine, the re-estimated chain
        // behind it, the job arc into the op after it), the row of the op that now follows it on the machine (new machine
        // predecessor), and the rows the one-step transients touch (this step's are the stepped op and that follower; the
        // previous step's revert).  Everything else is bit-identical to what is already there, so a lane emits at most two
        // rows (slot 0: its op of the stepped job, slot 1: one of the three extras) instead of ITER; an invalid action
        // changed nothing.
        const bool inc = (MODE & MODE_STEP) && P.obs_inc;
        const int row0 = (valid && gl >= apos && gl < M) ? ja * M + gl : -1;
        const int row1 = !valid ? -1 : gl == 0 ? o_next : gl == 1 ? rem_prev : gl == 2 ? fresh_prev : -1;
#pragma unroll
        for (int it = 0; it < ITER; it++) {
            if (inc && it >= 2) break;
            const int v = inc ? (it == 0 ? row0 : row1) : gl + it * G;
            if (v >= 0 && v < N && active) emit_row(v, (s_mach[v] >= 0) ? DUR(v) * PSEL(v) : PSEL(v));
        }
        if (inc) {
            if (P.mfea && valid && gl == 0) emit_mach(mc, o_tail);
        } else {
            // lane k = machine k: its route is the k-th range of the flat order, the tail its last entry
            const int c = (gl < M) ? (int)s_cnt[gl] : 0;
            int incs = c;
#pragma unroll
            for (int o = 1; o < G; o <<= 1) {
                const int n_ = __shfl_up_sync(FULL, incs, o, G);
                if (gl >= o) incs += n_;
            }
            if (P.mfea && gl < M && active) emit_mach(gl, c > 0 ? (int)s_ord[incs - 1] : 0);
        }
    }

    if (fr && active) {
        // The records were staged from the snapshot, not from the state: write them back whole, 16 bytes per lane (the
        // observation part above only reads them)
        const double2* s2 = reinterpret_cast<const double2*>(s_sd);
        double2* g2 = reinterpret_cast<double2*>(g_sd);
#pragma unroll 1
        for (int i = gl; i < S::SD / 2; i += G) g2[i] = s2[i];
        const int4* s4 = reinterpret_cast<const int4*>(s_si);
        int4* g4 = reinterpret_cast<int4*>(g_si);
#pragma unroll 1
        for (int i = gl; i < S::SI / 8; i += G) g4[i] = s4[i];
    }
    if (OVL && P.ep) {  // the entry index wb0 / EPW is recomputed rather than kept live through the step
        __syncwarp();
        if ((threadIdx.x & 31) == 0) {
            const unsigned bk = P.rev ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
            ovl_release(P.done_ep + bk * S::WARPS + (threadIdx.x >> 5), P.ep);
        }
    }
}

// ---- static tables: min feasible duration / energy per op, edge id per machine ----
__global__ void load_kernel(Layout L, const double* __restrict__ t, const double* __restrict__ p,
                            const double* __restrict__ tt, const int32_t* __restrict__ edge, int W, double* xs,
                            int8_t* edge_id) {
    size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)L.B * L.N;
    if (gid < total) {
        size_t b = gid / L.N;
        int i = (int)(gid % L.N);
        const double* tr = t + gid * L.M;
        const double* pr = p + gid * L.M;
        double mn = INFINITY, mnpt = INFINITY;
        for (int m = 0; m < L.M; m++) {  // SS:1932-1950
            double tv = tr[m], ptv = tv * fabs(pr[m]);
            if (!(tv < 0) && tv < mn) mn = tv;
            if (!(ptv < 0) && ptv < mnpt) mnpt = ptv;
        }
        xs[b * L.xs_stride + L.o_mind + i] = mn;
        xs[b * L.xs_stride + L.o_minpt + i] = mnpt;
    }
    size_t ntt = (size_t)L.B * L.M * L.M;
    if (gid < ntt) {
        size_t b = gid / (L.M * L.M);
        int r = (int)(gid % (L.M * L.M));
        xs[b * L.xs_stride + L.o_tt + r] = tt[gid];
    }
    if (gid < (size_t)L.B * L.M) {
        size_t b = gid / L.M;
        int m = (int)(gid % L.M);
        int id = 0;
        for (int g = 0; g < L.E && id == 0; g++)
            for (int k = 0; k < W; k++)
                if (edge[(b * L.E + g) * W + k] == m) { id = g + 1; break; }
        edge_id[gid] = (int8_t)id;
    }
}

// Synthetic instances on the device (reference distributions: instance/generate_allsize_mofjsp_dataset.py:161-273 with
// instance/config_ins.json's ranges): per op a mean time U(1,99) and mean power U(1,20), per (op, machine) multiplicative
// noise U(0.8,1.2); k ~ randint(0, M) machines of the op chosen without replacement (partial Fisher-Yates) are made
// infeasible by negating t and p; tt symmetric, zero diagonal, U(1,10) inside an edge group and U(10 d, 20 d) across
// groups at distance d; machines split contiguously into E groups (last group takes the remainder, padded with -1).
// Counter-based: every draw is a function of (seed, global env index, op / machine pair, draw number), so any slice of a
// batch can be generated on any rank.  One thread per (env, op) for t / p; the first M * M threads of an env also fill tt
// and the first E * W the edge table.
__device__ __forceinline__ double u01(uint64_t seed, uint64_t env, uint64_t item, uint64_t k) {
    const uint64_t x = splitmix64(seed ^ splitmix64(env * 0x100000001B3ULL + item * 0x9E3779B97F4A7C15ULL + k * 0xD1B54A32D192ED03ULL));
    return (double)(x >> 11) * (1.0 / 9007199254740992.0);  // 53 bits -> [0, 1)
}

__global__ void instance_gen_kernel(int B, int J, int M, int E, int W, uint64_t seed, uint64_t env_offset, double* t, double* p,
                                    double* tt, int32_t* edge) {
    const int N = J * M;
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)B * N) return;
    const size_t b = gid / N;
    const int i = (int)(gid % N);
    const uint64_t env = env_offset + b;
    {
        const double avg_t = 1.0 + 98.0 * u01(seed, env, i, 0), avg_p = 1.0 + 19.0 * u01(seed, env, i, 1);
        int k = (int)(u01(seed, env, i, 2) * M);  // 0 .. M-1 infeasible machines: at least one stays feasible
        if (k > M - 1) k = M - 1;
        unsigned char perm[64];
        for (int m = 0; m < M; m++) perm[m] = (unsigned char)m;
        uint64_t neg = 0;
        for (int q = 0; q < k; q++) {  // choose k of M without replacement
            int r = q + (int)(u01(seed, env, i, 3 + q) * (M - q));
            if (r > M - 1) r = M - 1;
            const unsigned char tmp = perm[q]; perm[q] = perm[r]; perm[r] = tmp;
            neg |= 1ull << perm[q];
        }
        for (int m = 0; m < M; m++) {
            double tv = avg_t * (0.8 + 0.4 * u01(seed, env, i, 100 + m));
            double pv = avg_p * (0.8 + 0.4 * u01(seed, env, i, 200 + m));
            if ((neg >> m) & 1) { tv = -tv; pv = -pv; }
            t[gid * M + m] = tv;
            p[gid * M + m] = pv;
        }
    }
    const int avg = M / E;
    auto group_of = [&](int m) { const int g = m / (avg > 0 ? avg : 1); return g < E - 1 ? g : E - 1; };
    if (i < M * M) {
        const int r = i / M, c = i % M;
        double v = 0.0;
        if (r != c) {
            const int lo = r < c ? r : c, hi = r < c ? c : r;  // one draw per unordered pair: symmetric
            const int dgrp = abs(group_of(lo) - group_of(hi));
            const double u = u01(seed, env, (uint64_t)N + (uint64_t)lo * M + hi, 0);
            v = dgrp == 0 ? 1.0 + 9.0 * u : 10.0 * dgrp + 10.0 * dgrp * u;
        }
        tt[(b * M + r) * M + c] = v;
    }
    if (i < E * W) {
        const int g = i / W, k2 = i % W;
        const int start = g * avg, size = g < E - 1 ? avg : M - avg * (E - 1);
        edge[(b * E + g) * W + k2] = k2 < size ? start + k2 : -1;
    }
}

__global__ void scaler_kernel(Layout L, double* sd, int full) {
    size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int per = full ? 13 : 4;
    if (gid < (size_t)L.B * per) {
        size_t b = gid / per;
        int k = (int)(gid % per);
        sd[b * L.sd_stride + L.o_sc + k] = 0.0;
    }
}

// cal_cur_task_machine_feature, trainer/parallel_env.py:152-214.  One thread per env.
template <typename OutT>
__global__ void mfea1_kernel(Layout L, const double* __restrict__ t, const double* __restrict__ p,
                             const double* __restrict__ xs, const int16_t* __restrict__ si,
                             const int8_t* __restrict__ edge_id, const int32_t* __restrict__ op, OutT* out,
                             uint8_t* mmask) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= L.B) return;
    const int M = L.M, N = L.N;
    int a = op[b];
    if (a < 0 || a >= N) {
        for (int m = 0; m < M; m++) {
            for (int k = 0; k < 6; k++) out[((size_t)b * M + m) * 6 + k] = (OutT)0;
            if (mmask) mmask[(size_t)b * M + m] = 1;
        }
        return;
    }
    const double* tr = t + ((size_t)b * N + a) * M;
    const double* pr = p + ((size_t)b * N + a) * M;
    double tv[64], ptv[64], pv[64];
    int nt = 0, npt = 0, npp = 0;
    for (int m = 0; m < M; m++) {
        double tm = tr[m], pm = pr[m], ptm = tm * fabs(pm);
        if (tm > 0) tv[nt++] = tm;
        if (ptm > 0) ptv[npt++] = ptm;
        if (pm > 0) pv[npp++] = pm;
    }
    double mean_t = np_sum_small(tv, nt) / (double)nt;
    double mean_pt = np_sum_small(ptv, npt) / (double)npt;
    double mean_p = np_sum_small(pv, npp) / (double)npp;
    int pm_row = M - 1;  // int(tfea[a-1][5]) - 1 wraps to the last row while the predecessor is unscheduled
    if (a % M != 0) {
        int mp = si[(size_t)b * L.si_stride + L.o_mach + a - 1];
        if (mp >= 0) pm_row = mp;
    }
    const double* ttrow = xs + (size_t)b * L.xs_stride + L.o_tt + pm_row * M;
    for (int m = 0; m < M; m++) {
        double tm = tr[m], pm = pr[m], ptm = tm * fabs(pm);
        int infeasible = !(tm >= 0);
        OutT* f = out + ((size_t)b * M + m) * 6;
        f[0] = (OutT)(tm > 0 ? tm : mean_t);
        f[1] = (OutT)(ptm > 0 ? ptm : mean_pt);
        f[2] = (OutT)((a % M == 0) ? 0.0 : ttrow[m]);
        f[3] = (OutT)(1 - infeasible);
        f[4] = (OutT)(pm > 0 ? pm : mean_p);
        f[5] = (OutT)edge_id[(size_t)b * M + m];
        if (mmask) mmask[(size_t)b * M + m] = (uint8_t)infeasible;
    }
}

// uniform random valid action from the current masks; one thread per env
__global__ void policy_kernel(Layout L, const double* __restrict__ t, const int16_t* __restrict__ si,
                              const uint8_t* __restrict__ jm, const int32_t* __restrict__ cand, uint64_t seed,
                              uint64_t env_offset, int32_t* op, int32_t* mach) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= L.B) return;
    const int J = L.J, M = L.M;
    const uint8_t* mk = jm + (size_t)b * J;
    int n = 0;
    for (int j = 0; j < J; j++) n += !mk[j];
    if (n == 0) { op[b] = -1; mach[b] = -1; return; }
    uint64_t step = (uint64_t)si[(size_t)b * L.si_stride + L.o_misc + 2];
    int k = (int)(((uint64_t)rand_u32(seed, env_offset + b, step, 0) * (uint64_t)n) >> 32);
    int a = -1;
    for (int j = 0; j < J; j++)
        if (!mk[j]) {
            if (k == 0) { a = cand[(size_t)b * J + j]; break; }
            k--;
        }
    const double* tr = t + ((size_t)b * L.N + a) * M;
    int nf = 0;
    for (int m = 0; m < M; m++) nf += (tr[m] >= 0);
    int km = (int)(((uint64_t)rand_u32(seed, env_offset + b, step, 1) * (uint64_t)nf) >> 32);
    int mm = -1;
    for (int m = 0; m < M; m++)
        if (tr[m] >= 0) {
            if (km == 0) { mm = m; break; }
            km--;
        }
    op[b] = a;
    mach[b] = mm;
}

// Size-templated pre-step kernel: (optionally) the random policy and the candidate-machine features of the
// chosen op in one pass; the op's t / p rows are read once into registers.  One thread per env.
template <int M, typename OutT, bool POLICY>
__global__ void __launch_bounds__(128) prestep_kernel(Layout L, const double* __restrict__ t, const double* __restrict__ p,
                                                      const double* __restrict__ xs, const int16_t* __restrict__ si,
                                                      const int8_t* __restrict__ edge_id, const uint8_t* __restrict__ jm,
                                                      const int32_t* __restrict__ cand, uint64_t seed, uint64_t env_offset,
                                                      int32_t* op, int32_t* mach, OutT* out, uint8_t* mmask) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= L.B) return;
    const int N = L.N, J = L.J;
    int a;
    uint64_t step = 0;
    if (POLICY) {
        const uint8_t* mk = jm + (size_t)b * J;
        int n = 0;
        for (int j = 0; j < J; j++) n += !mk[j];
        if (n == 0) { op[b] = -1; mach[b] = -1; return; }
        step = (uint64_t)si[(size_t)b * L.si_stride + L.o_misc + 2];
        int k = (int)(((uint64_t)rand_u32(seed, env_offset + b, step, 0) * (uint64_t)n) >> 32);
        a = -1;
        for (int j = 0; j < J; j++)
            if (!mk[j]) {
                if (k == 0) { a = cand[(size_t)b * J + j]; break; }
                k--;
            }
        op[b] = a;
    } else {
        a = op[b];
    }
    const bool bad = a < 0 || a >= N;
    const int ar = bad ? 0 : a;
    double tr[M], pr[M];
    {
        const double* trow = t + ((size_t)b * N + ar) * M;
        const double* prow = p + ((size_t)b * N + ar) * M;
        if constexpr (M % 2 == 0) {
#pragma unroll
            for (int m = 0; m < M; m += 2) {
                const double2 tv = __ldg(reinterpret_cast<const double2*>(trow + m));
                const double2 pv = __ldg(reinterpret_cast<const double2*>(prow + m));
                tr[m] = tv.x; tr[m + 1] = tv.y; pr[m] = pv.x; pr[m + 1] = pv.y;
            }
        } else {
#pragma unroll
            for (int m = 0; m < M; m++) { tr[m] = __ldg(trow + m); pr[m] = __ldg(prow + m); }
        }
    }
    if (POLICY) {
        int nf = 0;
#pragma unroll
        for (int m = 0; m < M; m++) nf += (tr[m] >= 0);
        int km = (int)(((uint64_t)rand_u32(seed, env_offset + b, step, 1) * (uint64_t)nf) >> 32);
        int mm = -1;
#pragma unroll
        for (int m = 0; m < M; m++)
            if (tr[m] >= 0) {
                if (km == 0 && mm < 0) mm = m;
                km--;
            }
        mach[b] = mm;
    }
    if (!out) return;
    if (bad) {
        for (int k = 0; k < M * 6; k++) out[(size_t)b * M * 6 + k] = (OutT)0;
        if (mmask)
            for (int m = 0; m < M; m++) mmask[(size_t)b * M + m] = 1;
        return;
    }
    // means over the positive entries, numpy pairwise order on the compacted row (parallel_env.py:177-184)
    double ct[M], cpt[M], cp[M];
    int nt = 0, npt = 0, npp = 0;
#pragma unroll
    for (int m = 0; m < M; m++) {
        const double ptm = tr[m] * fabs(pr[m]);
        if (tr[m] > 0) ct[nt++] = tr[m];
        if (ptm > 0) cpt[npt++] = ptm;
        if (pr[m] > 0) cp[npp++] = pr[m];
    }
    const double mean_t = np_sum_small(ct, nt) / (double)nt;
    const double mean_pt = np_sum_small(cpt, npt) / (double)npt;
    const double mean_p = np_sum_small(cp, npp) / (double)npp;
    int pm_row = M - 1;  // int(tfea[a-1][5]) - 1 wraps to the last row while the predecessor is unscheduled
    if (a % M != 0) {
        const int mp = si[(size_t)b * L.si_stride + L.o_mach + a - 1];
        if (mp >= 0) pm_row = mp;
    }
    const double* ttrow = xs + (size_t)b * L.xs_stride + L.o_tt + pm_row * M;
    OutT f[M * 6];
    uint8_t msk[M];
#pragma unroll
    for (int m = 0; m < M; m++) {
        const double tm = tr[m], pm = pr[m], ptm = tm * fabs(pm);
        const int infeasible = !(tm >= 0);
        f[m * 6 + 0] = (OutT)(tm > 0 ? tm : mean_t);
        f[m * 6 + 1] = (OutT)(ptm > 0 ? ptm : mean_pt);
        f[m * 6 + 2] = (OutT)((a % M == 0) ? 0.0 : __ldg(ttrow + m));
        f[m * 6 + 3] = (OutT)(1 - infeasible);
        f[m * 6 + 4] = (OutT)(pm > 0 ? pm : mean_p);
        f[m * 6 + 5] = (OutT)edge_id[(size_t)b * M + m];
        msk[m] = (uint8_t)infeasible;
    }
    OutT* o = out + (size_t)b * M * 6;
    if constexpr ((M * 6 * sizeof(OutT)) % 16 == 0) {
        constexpr int PER = 16 / sizeof(OutT);
        uint4* o4 = reinterpret_cast<uint4*>(o);
#pragma unroll
        for (int k = 0; k < M * 6 / PER; k++) o4[k] = *reinterpret_cast<const uint4*>(&f[k * PER]);
    } else {
#pragma unroll
        for (int k = 0; k < M * 6; k++) o[k] = f[k];
    }
    if (mmask) {
#pragma unroll
        for (int m = 0; m < M; m++) mmask[(size_t)b * M + m] = msk[m];
    }
}

template <typename OutT>
__global__ void dense_adj_kernel(Layout L, const float* __restrict__ adj_w, const int16_t* __restrict__ adj_src,
                                 OutT* adj) {
    // one block per env row-chunk: zero-fill then scatter (<= 3 entries per row)
    size_t b = blockIdx.x;
    const int N = L.N;
    OutT* A = adj + b * (size_t)N * N;
    for (size_t i = threadIdx.x; i < (size_t)N * N; i += blockDim.x) A[i] = (OutT)0;
    __syncthreads();
    for (int v = threadIdx.x; v < N; v += blockDim.x) {
        A[(size_t)v * N + v] = (OutT)1;
        float wj = adj_w[(b * N + v) * 2], wm = adj_w[(b * N + v) * 2 + 1];
        int src = adj_src[b * N + v];
        if (wj != 0.f) A[(size_t)v * N + v - 1] = (OutT)wj;
        if (src >= 0) A[(size_t)v * N + src] = (OutT)wm;
    }
}

// Raw arc weights of the disjunctive graph between real ops: out[b][u][v] = trunc(weight of arc u -> v), 0 = no arc --
// what nx.to_numpy_array(G)[1:-1, 1:-1].astype(int) holds in the reference (SS:2019) and what its gym `state` vector is
// made of (SS:2075-2130).  Same arc rules as the observation rows of env_kernel (job arc refresh SS:1356-1434, the
// machine arcs of SS:1548-1765, the one-step transients); compatibility view of the single-env class, not on the hot path.
// One thread per (env, destination op); the caller zero-fills `out`.
__global__ void raw_adj_kernel(Layout L, const double* __restrict__ sd, const int16_t* __restrict__ si,
                               const double* __restrict__ xs, int32_t* out) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)L.B * L.N) return;
    const size_t b = gid / L.N;
    const int v = (int)(gid % L.N), N = L.N, M = L.M;
    const double* d = sd + b * L.sd_stride;
    const int16_t* q = si + b * L.si_stride;
    const double* tt = xs + b * L.xs_stride + L.o_tt;
    const int rem_head = q[L.o_misc + 0], fresh = q[L.o_misc + 1];
    const int mv = q[L.o_mach + v];
    const bool sch = mv >= 0, vfirst = (v % M) == 0;
    const int rp = sch ? (int)q[L.o_rpred + v] : -1;
    const bool has_job = !vfirst && v != rem_head;
    const bool co = has_job && rp == v - 1;
    const bool has_m = rp >= 0 && !co;
    int32_t* A = out + b * (size_t)N * N;
    if (has_job) {
        const int u = v - 1, mu = q[L.o_mach + u];
        const double du = d[L.o_dur + u];
        double w;
        if (fresh == v) w = du + tt[mu * M + mv] + (d[L.o_st + v] - d[L.o_ft + u]);
        else if (du != 0.0) w = du + ((mu >= 0 && sch) ? tt[mu * M + mv] : 0.0);
        else w = 1.0;
        A[(size_t)u * N + v] = (int32_t)(long long)w;
    }
    if (has_m) {
        const double w = d[L.o_dur + rp] + ((rp / M == v / M) ? tt[mv * M + mv] : 0.0) + (d[L.o_st + v] - d[L.o_ft + rp]);
        A[(size_t)rp * N + v] = (int32_t)(long long)w;
    }
}

__global__ void export_kernel(Layout L, const double* __restrict__ sd, const int16_t* __restrict__ si, int32_t* mach,
                              double* st, double* ft, int32_t* routes) {
    size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (size_t)L.B * L.N) return;
    size_t b = gid / L.N;
    int i = (int)(gid % L.N);
    int mv = si[b * L.si_stride + L.o_mach + i];
    if (mach) mach[gid] = mv;
    if (st) st[gid] = mv >= 0 ? sd[b * L.sd_stride + L.o_st + i] : 0.0;
    if (ft) ft[gid] = mv >= 0 ? sd[b * L.sd_stride + L.o_ft + i] : 0.0;
    if (routes && i < L.M) {  // thread (b, m): machine m's route is its range of the flat order
        const int16_t* q = si + b * L.si_stride;
        int off = 0;
        for (int k = 0; k < i; k++) off += q[L.o_cnt + k];
        const int c = q[L.o_cnt + i];
        for (int k = 0; k < c; k++) routes[(b * L.M + i) * L.N + k] = q[L.o_ord + off + k];
    }
}

__global__ void fill_i32_kernel(int32_t* p, size_t n, int32_t v) {
    size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid < n) p[gid] = v;
}

__global__ void costs_kernel(Layout L, const double* __restrict__ sd, double* cost4, double* total_e1) {
    size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= (size_t)L.B) return;
    const double* s = sd + b * L.sd_stride + L.o_scal;
    if (cost4) {
        cost4[b * 4 + 0] = s[0];
        cost4[b * 4 + 1] = s[1] / (double)L.N;
        cost4[b * 4 + 2] = s[2];
        cost4[b * 4 + 3] = s[3];
    }
    if (total_e1) total_e1[b] = s[1];
}

__global__ void export_scaler_kernel(Layout L, const double* __restrict__ sd, double* R, double* mean, double* S,
                                     int64_t* n) {
    size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= (size_t)L.B) return;
    const double* s = sd + b * L.sd_stride + L.o_sc;
    for (int k = 0; k < 4; k++) { R[b * 4 + k] = s[k]; mean[b * 4 + k] = s[4 + k]; S[b * 4 + k] = s[8 + k]; }
    n[b] = (int64_t)s[12];
}

// Episode reset from the snapshot of the first one: the reset image of an env (initial estimates, counters, links,
// initial makespan / energy estimates) depends on the instance only, so later resets are one coalesced copy of the env
// part of `sd` (everything in front of the reward-scaler block; the three reward weights come from the caller), the
// whole `si` record and the initial job masks / candidates -- instead of re-deriving them per env.  One block per env,
// 16 bytes per thread (records are 16-byte aligned).
__global__ void reset_copy_kernel(Layout L, const double* __restrict__ sd0, const int16_t* __restrict__ si0,
                                  const double* __restrict__ weights, double* __restrict__ sd, int16_t* __restrict__ si,
                                  uint8_t* __restrict__ jm_fin, uint8_t* __restrict__ jm_esa, int32_t* __restrict__ cand) {
    const size_t b = blockIdx.x;
    const double2* src = reinterpret_cast<const double2*>(sd0 + b * L.sd_stride);
    double2* dst = reinterpret_cast<double2*>(sd + b * L.sd_stride);
    auto word = [&](const int i, const double v) { return (i >= L.o_w && i < L.o_w + 3) ? weights[b * 3 + (i - L.o_w)] : v; };
    for (int k = threadIdx.x; 2 * k < L.o_sc; k += blockDim.x) {  // the part in front of the reward-scaler block
        const double2 v = src[k];
        if (2 * k + 1 < L.o_sc) dst[k] = make_double2(word(2 * k, v.x), word(2 * k + 1, v.y));
        else sd[b * L.sd_stride + 2 * k] = word(2 * k, v.x);
    }
    const int4* si_src = reinterpret_cast<const int4*>(si0 + b * L.si_stride);
    int4* si_dst = reinterpret_cast<int4*>(si + b * L.si_stride);
    for (int k = threadIdx.x; k < L.si_stride / 8; k += blockDim.x) si_dst[k] = si_src[k];
    for (int j = threadIdx.x; j < L.J; j += blockDim.x) {
        jm_fin[b * L.J + j] = 0;
        jm_esa[b * L.J + j] = 0;
        cand[b * L.J + j] = j * L.M;
    }
}

// Env gather (mtfjsp_gather): destination env b becomes a copy of source env idx[b] -- every per-env record and table the
// handle keeps.  The two handles share (J, M, E), so they share every stride.
struct GatherArgs {
    Layout L;
    int src_B;
    const int32_t* idx;
    const double *sd, *sd0, *xs, *t, *p;
    const int16_t *si, *si0;
    const int8_t* edge_id;
    const uint8_t *jm_fin, *jm_esa, *dn, *inv;
    const int32_t* cand;
    double *d_sd, *d_sd0, *d_xs, *d_t, *d_p;
    int16_t *d_si, *d_si0;
    int8_t* d_edge_id;
    uint8_t *d_jm_fin, *d_jm_esa, *d_dn, *d_inv;
    int32_t* d_cand;
};

template <typename W>
__device__ __forceinline__ void copy_words(void* dst, const void* src, size_t n) {
    for (size_t k = threadIdx.x; k < n; k += blockDim.x) reinterpret_cast<W*>(dst)[k] = reinterpret_cast<const W*>(src)[k];
}

// One block per destination env, 16 bytes per thread (every record is 16-byte aligned; the t / p tables of one env are
// too when N*M is even, 8-byte words otherwise), as reset_copy_kernel.  A source index outside the batch is input from
// outside the program: that env gets its invalid flag and nothing else.
__global__ void __launch_bounds__(128) gather_kernel(const __grid_constant__ GatherArgs A) {
    const Layout& L = A.L;
    const size_t b = blockIdx.x;
    const int src = A.idx[b];
    if (src < 0 || src >= A.src_B) {
#ifdef MTFJSP_DEBUG_BOUNDS  // debug builds: an out-of-range source env is a caller bug worth stopping at
        assert(src >= 0 && src < A.src_B);
#endif
        if (threadIdx.x == 0) A.d_inv[b] = 1;
        return;
    }
    const size_t a = (size_t)src;
    copy_words<double2>(A.d_sd + b * L.sd_stride, A.sd + a * L.sd_stride, L.sd_stride / 2);
    copy_words<double2>(A.d_sd0 + b * L.sd_stride, A.sd0 + a * L.sd_stride, L.sd_stride / 2);
    copy_words<double2>(A.d_xs + b * L.xs_stride, A.xs + a * L.xs_stride, L.xs_stride / 2);
    copy_words<int4>(A.d_si + b * L.si_stride, A.si + a * L.si_stride, L.si_stride / 8);
    copy_words<int4>(A.d_si0 + b * L.si_stride, A.si0 + a * L.si_stride, L.si_stride / 8);
    const size_t nm = (size_t)L.N * L.M;
    if (nm % 2 == 0) {
        copy_words<double2>(A.d_t + b * nm, A.t + a * nm, nm / 2);
        copy_words<double2>(A.d_p + b * nm, A.p + a * nm, nm / 2);
    } else {
        copy_words<double>(A.d_t + b * nm, A.t + a * nm, nm);
        copy_words<double>(A.d_p + b * nm, A.p + a * nm, nm);
    }
    for (int k = threadIdx.x; k < L.M; k += blockDim.x) A.d_edge_id[b * L.M + k] = A.edge_id[a * L.M + k];
    for (int j = threadIdx.x; j < L.J; j += blockDim.x) {
        A.d_jm_fin[b * L.J + j] = A.jm_fin[a * L.J + j];
        A.d_jm_esa[b * L.J + j] = A.jm_esa[a * L.J + j];
        A.d_cand[b * L.J + j] = A.cand[a * L.J + j];
    }
    if (threadIdx.x == 0) {
        A.d_dn[b] = A.dn[a];
        A.d_inv[b] = A.inv[a];
    }
}

// bytes gather_kernel copies per env (each read once and written once)
size_t gather_env_bytes(const Layout& L) {
    return (size_t)2 * L.sd_stride * 8 + (size_t)L.xs_stride * 8 + (size_t)2 * L.si_stride * 2 + (size_t)2 * L.N * L.M * 8 +
           (size_t)L.M + (size_t)2 * L.J + (size_t)4 * L.J + 2;
}

// One-step lookahead (mtfjsp_peek): what mtfjsp_step would return for each of K (op, machine) pairs per env, computed
// from a read-only copy of the env's records.  One block per env stages the records once; then, per chunk of
// PEEK_CHUNK pairs, warps evaluate one pair each (placement scan, makespan, energy) and threads finish one pair each
// (the sequential idle sum and the reward).  Every quantity is the step's own FP64 expression in the step's operand
// order (env_kernel above), restated on the read-only copy by deltas:
//   placement  the step's scan over machine m's route, unchanged;
//   makespan   max over every op of its finish time, job a/M's remaining chain re-derived from a's new finish;
//   energy     numpy's pairwise sum of the per-op estimate with a's term d*p in place of minpt[a]: only the leaf that
//              holds a is re-added, the other leaves are the env's (computed once per block), then the leaves are
//              combined by the plan's postfix program;
//   idle time  the flat-order sequential sum: the unchanged prefix in front of a's slot (prefix sums computed once per
//              block), a's term, its route follower's term against a's new finish, then the unchanged rest.
// The idle term (idle_term), the per-op energy estimate (energy_est) and the reward (reward_terms) are the step's own
// device code.  The validity test, the placement scan, the leaf pass and the postfix fold stay restated here: shared
// with env_transition / pairwise_sum, each of them changed the SASS of the generic step and replay kernels and made the
// replay slower at J6M6 and J10M10.
struct PeekArgs {
    Layout L;
    PwPlan pw;
    const double *sd, *xs, *t, *p;
    const int16_t* si;
    const int32_t *op, *mach;
    int K;
    double cfgw[3], divisor;
    double* reward5;
    uint8_t* invalid;
};

constexpr int PEEK_CHUNK = 128, PEEK_STK = 16;

// shared-memory plan of peek_kernel (bytes): the staged record prefix st ft dur psel scal, the static doubles, the idle
// prefix sums, the base leaf results, the si record up to the counters and nsched, the route offsets, the per-warp leaf
// combine stacks and the per-pair results of one chunk
struct PeekSmem {
    int sd, xs, pre, leaf, stk, si, off, c_d, c_i, total;
};
__host__ __device__ inline PeekSmem peek_smem(const Layout& L, int nleaves, int warps) {
    PeekSmem s;
    int o = 0;
    s.sd = o; o += (L.o_scal + 4 + 1) / 2 * 16;
    s.xs = o; o += L.xs_stride * 8;
    s.pre = o; o += (L.N + 1) * 8;
    s.leaf = o; o += nleaves * 8;
    s.stk = o; o += warps * PEEK_STK * 8;
    s.c_d = o; o += PEEK_CHUNK * 5 * 8;  // st, d, mk, env, trans per pair
    s.c_i = o; o += PEEK_CHUNK * 4 * 4;  // valid, slot, next, prev per pair
    s.si = o; o += (L.o_misc + 3) * 2;
    s.off = (o + 3) / 4 * 4; o = s.off + L.M * 4;
    s.total = (o + 15) / 16 * 16;
    return s;
}

// one leaf of numpy's pairwise sum (pairwise_sum's leaf pass) over est(off .. off + n - 1); every 8-lane segment
// computes it, lane k == 0 of a segment holds the result
template <class Est>
__device__ __forceinline__ double peek_leaf(const Est& est, int off, int n, int k) {
    const int nb = (n >= 8) ? n - (n & 7) : 0;
    double r = 0.0;
    if (n >= 8) {
        r = est(off + k);
        for (int i = 8 + k; i < nb; i += 8) r += est(off + i);
    }
    r = r + __shfl_down_sync(FULL, r, 1, 8);
    r = r + __shfl_down_sync(FULL, r, 2, 8);
    r = r + __shfl_down_sync(FULL, r, 4, 8);
    double res = r;
    if (k == 0)
        for (int i = nb; i < n; i++) res += est(off + i);
    return res;
}

__global__ void __launch_bounds__(128) peek_kernel(const __grid_constant__ PeekArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Layout& L = A.L;
    const PwPlan& pw = A.pw;
    const int N = L.N, M = L.M, K = A.K;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const size_t b = blockIdx.x;
    const PeekSmem S = peek_smem(L, pw.nleaves, nwarps);
    double* s_sd = reinterpret_cast<double*>(smem_raw + S.sd);
    double* s_xs = reinterpret_cast<double*>(smem_raw + S.xs);
    double* s_pre = reinterpret_cast<double*>(smem_raw + S.pre);
    double* s_leaf = reinterpret_cast<double*>(smem_raw + S.leaf);
    double* s_stk = reinterpret_cast<double*>(smem_raw + S.stk) + warp * PEEK_STK;
    double* c_d = reinterpret_cast<double*>(smem_raw + S.c_d);
    int* c_i = reinterpret_cast<int*>(smem_raw + S.c_i);
    int16_t* s_si = reinterpret_cast<int16_t*>(smem_raw + S.si);
    int* s_off = reinterpret_cast<int*>(smem_raw + S.off);

    // ---- stage the record prefix (st ft dur psel scal), the static doubles and the si record ----
    {
        const double* g_sd = A.sd + b * L.sd_stride;
        for (int i = threadIdx.x; i < L.o_scal + 4; i += blockDim.x) s_sd[i] = g_sd[i];
        const uint4* src = reinterpret_cast<const uint4*>(A.xs + b * L.xs_stride);
        uint4* dst = reinterpret_cast<uint4*>(s_xs);
        for (int i = threadIdx.x; i < L.xs_stride / 2; i += blockDim.x) dst[i] = __ldg(src + i);
        const int16_t* g_si = A.si + b * L.si_stride;
        for (int i = threadIdx.x; i < L.o_misc + 3; i += blockDim.x) s_si[i] = g_si[i];
    }
    __syncthreads();
    const double* s_st = s_sd + L.o_st;
    const double* s_ft = s_sd + L.o_ft;
    const double* s_dur = s_sd + L.o_dur;
    const double* s_psel = s_sd + L.o_psel;
    const double* s_scal = s_sd + L.o_scal;  // mk_prev, e_prev, trans, idle_prev
    const int16_t* s_mach = s_si + L.o_mach;
    const int16_t* s_ord = s_si + L.o_ord;
    const int16_t* s_rpred = s_si + L.o_rpred;
    const int16_t* s_cnt = s_si + L.o_cnt;
    const int nsched0 = s_si[L.o_misc + 2];
    const double* s_mind = s_xs + L.o_mind;
    const double* s_minpt = s_xs + L.o_minpt;
    const double* s_tt = s_xs + L.o_tt;
    // the env's per-op energy estimate (env_kernel's s_pt)
    const auto est = [&](int v) { return energy_est(s_mach, s_dur, s_psel, s_minpt, v); };
    if (warp == 0) {  // base leaf results, four leaves at a time as pairwise_sum
        for (int L0 = 0; L0 < pw.nleaves; L0 += 4) {
            const int Lx = L0 + (lane >> 3);
            const bool act = Lx < pw.nleaves;
            const double r = peek_leaf(est, act ? pw.leaf_off[Lx] : 0, act ? pw.leaf_len[Lx] : 0, lane & 7);
            if (act && (lane & 7) == 0) s_leaf[Lx] = r;
        }
    } else if (warp == 1) {  // route offsets: machine m's route is ord[off[m], off[m] + cnt[m])
        if (lane == 0) {
            int o = 0;
            for (int mm = 0; mm < M; mm++) { s_off[mm] = o; o += s_cnt[mm]; }
        }
    }
    if (threadIdx.x == 0) {  // idle prefix sums over the flat order: s_pre[g] = the step's running sum in front of term g
        double idle = 0.0;
        for (int g = 0; g < nsched0; g++) {
            s_pre[g] = idle;
            idle = idle + idle_term(s_st, s_ft, s_ord, s_rpred, g) * 1.0;
        }
        s_pre[nsched0] = idle;
    }
    __syncthreads();

    for (int k0 = 0; k0 < K; k0 += PEEK_CHUNK) {
        const int kn = min(PEEK_CHUNK, K - k0);
        // ---- phase 1: one warp per pair ----
        for (int c = warp; c < kn; c += nwarps) {
            const int a = A.op[b * K + k0 + c], m = A.mach[b * K + k0 + c];
            double d = 0.0, pa = 0.0;
            bool valid = (a >= 0) && (a < N) && (m >= 0) && (m < M) && (nsched0 < N);
            if (valid) valid = (s_mach[a] < 0) && (((a % M) == 0) || (s_mach[a - 1] >= 0));
            if (valid) {
                d = __ldg(A.t + (b * N + a) * M + m);
                pa = __ldg(A.p + (b * N + a) * M + m);
                valid = !(d < 0);
            }
            if (!valid) {
                if (lane == 0) c_i[c * 4] = 0;
                continue;
            }
            const bool first = (a % M) == 0;
            const int ja = a / M;
            // placement: env_kernel's scan over machine m's route (SS:1548-1601, 1689-1775)
            const double arr_a = first ? 0.0 : s_ft[a - 1] + s_tt[s_mach[a - 1] * M + m];
            const int len = s_cnt[m];
            const double ttmm = s_tt[m * M + m];
            const int offm = s_off[m];
            double st = arr_a;
            int where = 0, prev = -1, next = -1;
            if (len > 0) {
                const double lbft = arr_a + d;
                unsigned best = 0xffffffffu;
                const int lastop = s_ord[offm + len - 1];
                if (L.left_shift) {
                    for (int kk0 = 0; kk0 < len; kk0 += 32) {
                        const int kk = kk0 + lane;
                        unsigned key = 0xffffffffu;
                        if (kk < len) {
                            const int v = s_ord[offm + kk];
                            const bool vfirst = (v % M) == 0;
                            double nst = vfirst ? 0.0 : s_ft[v - 1] + s_tt[s_mach[v - 1] * M + m];
                            bool ok;
                            if (kk == 0) {
                                ok = (lbft <= nst);
                            } else {
                                const int rp = s_ord[offm + kk - 1];
                                double val = s_ft[rp] + ((rp / M == v / M) ? ttmm : 0.0);
                                nst = fmax(nst, val);
                                ok = !(lbft > nst) && !((nst - s_ft[rp]) < d);
                            }
                            if (ok) key = ((unsigned)kk << 16) | (unsigned)v;
                        }
                        best = min(best, __reduce_min_sync(FULL, key));
                    }
                }
                if (best != 0xffffffffu) {
                    where = (int)(best >> 16);
                    next = (int)(best & 0xffffu);
                    if (where > 0) {
                        prev = s_rpred[next];
                        double y = s_ft[prev] + ((prev / M == ja) ? ttmm : 0.0);
                        st = (y > arr_a) ? y : arr_a;
                    }
                } else {
                    where = len;
                    prev = lastop;
                    double y = s_ft[prev] + ((prev / M == ja) ? ttmm : 0.0);
                    st = (y > arr_a) ? y : arr_a;
                }
            }
            // makespan estimate: a's job from a on is the re-derived chain (SS:1964-1995), every other op as it stands
            double cur = st + d, mx = cur;
            for (int cc = (a % M) + 1; cc < M; cc++) {
                cur = cur + s_mind[ja * M + cc];
                mx = fmax(mx, cur);
            }
            for (int v = lane; v < N; v += 32)
                if (v < a || v >= (ja + 1) * M) mx = fmax(mx, s_ft[v]);
            const double mkv = warp_max(mx);
            // energy estimate: re-add the leaf holding a, combine the leaves with the plan's postfix program
            const double ea = d * pa;
            const auto est_a = [&](int v) { return v == a ? ea : est(v); };
            int La = 0;
            while (La + 1 < pw.nleaves && pw.leaf_off[La + 1] <= a) La++;
            const double leaf_a = peek_leaf(est_a, pw.leaf_off[La], pw.leaf_len[La], lane & 7);
            double env = leaf_a;
            if (lane == 0 && pw.nleaves > 1) {
                int sp = 0;
                for (int i = 0; i < pw.nprog; i++) {
                    const int q = pw.prog[i];
                    if (q >= 0) {
                        s_stk[sp++] = (q == La) ? leaf_a : s_leaf[q];
                    } else {
                        s_stk[sp - 2] = s_stk[sp - 2] + s_stk[sp - 1];
                        sp--;
                    }
                }
                env = s_stk[0];
            }
            if (lane == 0) {
                const double nt = first ? 0.0 : s_tt[s_mach[a - 1] * M + m];  // SS:872-877
                double* r = c_d + c * 5;
                r[0] = st; r[1] = d; r[2] = mkv; r[3] = env; r[4] = s_scal[2] + nt;
                int* q = c_i + c * 4;
                q[0] = 1; q[1] = offm + where; q[2] = next; q[3] = prev;
            }
            __syncwarp();
        }
        __syncthreads();
        // ---- phase 2: one thread per pair: idle sum, reward (wrk_reward_function, SS:1066-1132) ----
        for (int c = threadIdx.x; c < kn; c += blockDim.x) {
            const size_t o = b * K + k0 + c;
            const int* q = c_i + c * 4;
            if (!q[0]) {
                if (A.reward5)
                    for (int i = 0; i < 5; i++) A.reward5[o * 5 + i] = 0.0;
                if (A.invalid) A.invalid[o] = 1;
                continue;
            }
            const double* r = c_d + c * 5;
            const double st = r[0], ft = st + r[1];
            const int slot = q[1], next = q[2], prev = q[3];
            double idle = s_pre[slot];
            idle = idle + ((prev < 0) ? (st - 0.0) : (st - s_ft[prev])) * 1.0;
            int g = slot;
            if (next >= 0) {
                idle = idle + (s_st[next] - ft) * 1.0;
                g++;
            }
            for (; g < nsched0; g++) idle = idle + idle_term(s_st, s_ft, s_ord, s_rpred, g) * 1.0;
            const StepReward w = reward_terms(s_scal, A.cfgw, N, r[2], r[3], r[4], idle);
            if (A.reward5) {
                double* r5 = A.reward5 + o * 5;
                r5[0] = w.total / A.divisor; r5[1] = w.r_t; r5[2] = w.r_idle; r5[3] = w.r_pt; r5[4] = w.r_tt;
            }
            if (A.invalid) A.invalid[o] = 0;
        }
        __syncthreads();
    }
}

// bytes peek_kernel reads and writes for one env and K pairs: the staged records once, per pair the pair, its t / p
// entries, 5 rewards and the flag
size_t peek_env_bytes(const Layout& L, int K) {
    return (size_t)(L.o_scal + 4) * 8 + (size_t)L.xs_stride * 8 + (size_t)(L.o_misc + 3) * 2 +
           (size_t)K * (8 + 16 + 5 * 8 + 1);
}

// Whole-episode replay (mtfjsp_replay): candidate r runs T (op, machine) actions from the episode start of env src[r]
// (the reset snapshot sd0 / si0) and leaves the costs, the summed rewards and the index of its first invalid action.
// One warp per candidate, in env_kernel's lane layout and shared-memory slice (Layout::sm_*), so every size the handle
// accepts fits: the warp stages the snapshot records and the static doubles once, then runs every transition on that
// copy with env_kernel's own device code (env_transition, env_estimates, env_reward; peek_kernel shares their idle_term,
// energy_est and reward_terms) and writes 4 + 5 doubles and an int.
// The actions are read 32 at a time, one (op, machine) pair per lane in one coalesced 256-byte read, and broadcast by
// shuffle.  Nothing of the handle is written.
struct ReplayArgs {
    Layout L;
    PwPlan pw;
    const double *sd0, *xs, *t, *p;
    const int16_t* si0;
    const int32_t *src, *actions;
    int R, T;
    double cfgw[3], divisor;
    double *cost4, *return5;
    int32_t* first_invalid;
};

__global__ void __launch_bounds__(256) replay_kernel(const __grid_constant__ ReplayArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Layout& L = A.L;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * L.warps_per_block + warp;
    if (r >= A.R) return;
    const int src = A.src[r];
    if (src < 0 || src >= L.B) {  // a source index is data: this candidate gets -2 and zero rows, the others run
        if (A.cost4 && lane < 4) A.cost4[(size_t)r * 4 + lane] = 0.0;
        if (A.return5 && lane < 5) A.return5[(size_t)r * 5 + lane] = 0.0;
        if (A.first_invalid && lane == 0) A.first_invalid[r] = -2;
        return;
    }
    const EnvSmem S(L, smem_raw + (size_t)warp * L.smem_per_warp);
    {
        const uint4* g = reinterpret_cast<const uint4*>(A.sd0 + (size_t)src * L.sd_stride);
        uint4* d = reinterpret_cast<uint4*>(S.sd);
        for (int i = lane; i < L.sd_stride / 2; i += 32) d[i] = __ldg(g + i);
        g = reinterpret_cast<const uint4*>(A.xs + (size_t)src * L.xs_stride);
        d = reinterpret_cast<uint4*>(S.xs);
        for (int i = lane; i < L.xs_stride / 2; i += 32) d[i] = __ldg(g + i);
        g = reinterpret_cast<const uint4*>(A.si0 + (size_t)src * L.si_stride);
        d = reinterpret_cast<uint4*>(S.si);
        for (int i = lane; i < L.si_stride / 8; i += 32) d[i] = __ldg(g + i);
    }
    __syncwarp();
    const int32_t* act = A.actions + (size_t)r * A.T * 2;
    double ret[5] = {0.0, 0.0, 0.0, 0.0, 0.0};  // lane 0: the step-order sums of the step's reward5
    int bad = -1, op_l = 0, mach_l = 0;
    for (int s = 0; s < A.T; s++) {
        if ((s & 31) == 0) {
            op_l = s + lane < A.T ? __ldg(act + 2 * (s + lane)) : 0;
            mach_l = s + lane < A.T ? __ldg(act + 2 * (s + lane) + 1) : 0;
        }
        const int a = __shfl_sync(FULL, op_l, s & 31), m = __shfl_sync(FULL, mach_l, s & 31);
        const StepOut so = env_transition<false>(L, S, A.t, A.p, (size_t)src, a, m, nullptr, nullptr, lane);
        double r5[5] = {0.0, 0.0, 0.0, 0.0, 0.0};  // what the step writes for an invalid action
        if (so.valid) {
            double mkv, env;
            env_estimates<true>(L, A.pw, S, lane, &mkv, &env);
            const StepReward rw = env_reward(L, S, A.cfgw, m, mkv, env, so, lane);
            r5[0] = rw.total / A.divisor; r5[1] = rw.r_t; r5[2] = rw.r_idle; r5[3] = rw.r_pt; r5[4] = rw.r_tt;
            __syncwarp();
        } else if (bad < 0) {
            bad = s;
        }
#pragma unroll
        for (int k = 0; k < 5; k++) ret[k] += r5[k];
    }
    if (lane == 0) {
        if (A.cost4) {  // costs_kernel's expressions
            double* c = A.cost4 + (size_t)r * 4;
            c[0] = S.scal[0]; c[1] = S.scal[1] / (double)L.N; c[2] = S.scal[2]; c[3] = S.scal[3];
        }
        if (A.return5)
            for (int k = 0; k < 5; k++) A.return5[(size_t)r * 5 + k] = ret[k];
        if (A.first_invalid) A.first_invalid[r] = bad;
    }
}

thread_local char g_err[512] = "";

int fail(int code, const char* msg, cudaError_t e = cudaSuccess) {
    if (e != cudaSuccess) snprintf(g_err, sizeof g_err, "%s: %s", msg, cudaGetErrorString(e));
    else snprintf(g_err, sizeof g_err, "%s", msg);
    return code;
}

int align_up(int x, int a) { return (x + a - 1) / a * a; }

void build_plan_rec(int off, int n, PwPlan& pw) {
    if (n <= 128) {
        pw.leaf_off[pw.nleaves] = off;
        pw.leaf_len[pw.nleaves] = n;
        pw.prog[pw.nprog++] = (signed char)pw.nleaves;
        pw.nleaves++;
    } else {
        int n2 = n / 2;
        n2 -= n2 % 8;
        build_plan_rec(off, n2, pw);
        build_plan_rec(off + n2, n - n2, pw);
        pw.prog[pw.nprog++] = -1;
    }
}

}  // namespace

struct mtfjsp_env {
    Layout L;
    PwPlan pw;
    int device;
    double cfgw[3], divisor, gamma;
    double *sd, *xs, *t, *p;
    double* sd0;   // reset snapshot of sd / si (taken after the first reset since the last load)
    int16_t* si0;
    bool reset_snap;
    // MTFJSP_FUSED_RESET (default on): once the snapshot exists, mtfjsp_reset (and an mtfjsp_scaler_reset behind it) only
    // record the reset here.  The next step launch of a specialised kernel performs it -- it stages the snapshot instead
    // of the state and writes its records back whole -- instead of a separate pass over the batch's state.  Every other
    // entry point first runs the recorded reset as reset_copy_kernel + scaler_kernel (flush_reset).
    int fused_reset;
    bool pend_reset, pend_scaler;
    const double* pend_w;  // the caller's [B,3] weights: valid until the next call on the handle (include/mtfjsp.h)
    int16_t* si;
    int8_t* edge_id;
    uint8_t *jm_fin, *jm_esa;
    int32_t* cand;
    // scratch for the host-step / random-step paths
    int32_t *a_op, *a_mach;
    double *r5, *s4, *info6;
    int2* act2;          // packed host-step actions
    unsigned char* rec;  // packed host-step records
    int rec_stride;
    uint8_t *dn, *inv;
    float* tmp_adj_w;
    int16_t* tmp_adj_src;
    bool loaded, reset_done, force_generic;
    // incremental observation (mtfjsp_set_obs_incremental): which output buffers currently mirror the env state
    bool obs_inc_enabled, obs_inc_allowed, obs_synced;
    const void* obs_ptrs[4];
    int obs_dtype;
    bool host_act_in_place;  // host step: actions read from mapped host memory in place (MTFJSP_HOST_ZEROCOPY=2), else copied in
    int fuse_policy;  // MTFJSP_FUSE_POLICY, read from the environment at create time (tests compare the settings)
    int flip;         // successive eager step launches walk the batch in opposite directions for L2 reuse (Params::rev)
    // The small records every launch starts from -- job masks, candidates, the si record (route order, counters) -- live
    // in one slab that step launches mark as an L2-persisting access window, so the loads at the head of a warp's
    // dependent chain hit L2 instead of DRAM although the batch's working set is larger than L2
    unsigned char* slab;
    size_t slab_bytes, window_bytes;
    int64_t launches;
    // MTFJSP_LAUNCH_OVERLAP (default on): whole-batch step launches of the size-specialised kernel may start while the
    // previous one finishes (programmatic dependent launch; see ovl_wait).  done_ep: one completion epoch per warp-sized
    // env range, released by every such launch whatever the setting; ep: the epoch of the last one issued.  ovl_err:
    // mapped host word a launch sets when its wait timed out (ovl_err_d: its device address)
    // ovl_chain: the handle's last operation was a step launch that released its epoch
    int launch_overlap;
    bool ovl_chain;
    unsigned long long* done_ep;
    unsigned long long ep;
    unsigned *ovl_err, *ovl_err_d;
};

#define CK(call, msg)                                            \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return fail(MTFJSP_E_CUDA, msg, e_); \
    } while (0)

static Params make_params(mtfjsp_env* h) {
    Params P;
    memset(&P, 0, sizeof P);
    P.L = h->L;
    P.pw = h->pw;
    P.sd = h->sd; P.si = h->si; P.xs = h->xs; P.t = h->t; P.p = h->p;
    P.cfgw[0] = h->cfgw[0]; P.cfgw[1] = h->cfgw[1]; P.cfgw[2] = h->cfgw[2];
    P.divisor = h->divisor; P.gamma = h->gamma;
    P.jm_fin = h->jm_fin; P.jm_esa = h->jm_esa; P.cand_int = h->cand;
    return P;
}

// Runs the reset that mtfjsp_reset / mtfjsp_scaler_reset recorded (mtfjsp_env::pend_reset), if any.
static int flush_reset(mtfjsp_env* h, cudaStream_t s) {
    const Layout& L = h->L;
    if (h->pend_reset || h->pend_scaler) h->ovl_chain = false;
    if (h->pend_reset) {
        reset_copy_kernel<<<L.B, 128, 0, s>>>(L, h->sd0, h->si0, h->pend_w, h->sd, h->si, h->jm_fin, h->jm_esa, h->cand);
        h->launches++;
        h->pend_reset = false;
        CK(cudaGetLastError(), "reset_copy_kernel");
    }
    if (h->pend_scaler) {
        const size_t n = (size_t)L.B * 4;
        scaler_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(L, h->sd, 0);
        h->launches++;
        h->pend_scaler = false;
        CK(cudaGetLastError(), "scaler_kernel");
    }
    return MTFJSP_OK;
}

// Head of every entry point that touches env state: selects the device and runs a recorded reset -- unless the call
// is a step that may perform the reset itself (launch_spec decides; every other launch path flushes).
static int enter(mtfjsp_env* h, cudaStream_t s, bool step = false) {
    if (*(volatile unsigned*)h->ovl_err)
        return fail(MTFJSP_E_CUDA, "a step launch waited more than 1 s for the previous one (launch overlap)");
    CK(cudaSetDevice(h->device), "cudaSetDevice");
    if (!step) h->ovl_chain = false;  // this call may write what a step reads: the next step waits for it in full
    return step ? MTFJSP_OK : flush_reset(h, s);
}

template <int MODE, typename OutT>
static int launch_env(mtfjsp_env* h, const Params& P, cudaStream_t s) {
    const Layout& L = h->L;
    int rc = flush_reset(h, s);
    if (rc != MTFJSP_OK) return rc;
    size_t smem = (size_t)L.smem_per_warp * L.warps_per_block;
    static thread_local int configured_dev = -1;
    static thread_local size_t configured_smem = 0;
    if (configured_dev != h->device || configured_smem < smem) {
        CK(cudaFuncSetAttribute(env_kernel<MODE, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "cudaFuncSetAttribute");
        configured_dev = h->device;
        configured_smem = smem;
    }
    int blocks = (L.B + L.warps_per_block - 1) / L.warps_per_block;
    env_kernel<MODE, OutT><<<blocks, L.warps_per_block * 32, smem, s>>>(P);
    h->launches++;
    h->ovl_chain = false;
    CK(cudaGetLastError(), "env_kernel launch");
    return MTFJSP_OK;
}

template <class S, int MODE, typename OutT>
static int launch_spec(mtfjsp_env* h, const Params& P, cudaStream_t s) {
    const Layout& L = h->L;
    if (L.sd_stride != S::SD || L.si_stride != S::SI || L.xs_stride != S::XS || L.o_sc != S::O_SC || L.o_misc != S::O_MISC ||
        L.o_eacc != S::O_EACC || L.o_eleaf != S::O_ELEAF || L.o_ipre != S::O_IPRE || L.nich != S::NICH || h->pw.nleaves != S::NLEAF)
        return fail(MTFJSP_E_STATE, "specialised kernel layout mismatch");
    if constexpr (!S::COLD && (MODE & MODE_STEP) && !(MODE & (MODE_HOST | MODE_FROM_RESET))) {
        if (h->pend_reset) {  // this step performs the recorded reset
            Params Q = P;
            Q.sd0 = h->sd0; Q.si0 = h->si0; Q.weights = h->pend_w; Q.clear_ret = h->pend_scaler ? 1 : 0;
            h->pend_reset = h->pend_scaler = false;
            return launch_spec<S, MODE | MODE_FROM_RESET, OutT>(h, Q, s);
        }
    }
    if constexpr (!(MODE & MODE_FROM_RESET)) {
        const int rc = flush_reset(h, s);
        if (rc != MTFJSP_OK) return rc;
    }
    const size_t smem = (size_t)S::WARPS * S::EPW * S::ENV_BYTES + (S::BAR_IN_PAD ? 0 : 16 * ((S::WARPS * 8 + 15) / 16));
    static thread_local int configured_dev = -1;
    if (configured_dev != h->device) {
        CK(cudaFuncSetAttribute(env_kernel_s<S, MODE, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
           "cudaFuncSetAttribute");
        configured_dev = h->device;
    }
    const int per_block = S::WARPS * S::EPW;
    const int blocks = (L.B + per_block - 1) / per_block;
    Params Q = P;
    if (MODE & MODE_STEP) {  // eager step launches alternate direction (see Params::rev)
        Q.rev = h->flip;
        h->flip ^= 1;
    }
    // Launch overlap (ovl_wait).  Whole-batch step launches release epochs (Q.ep).  Only a random step without a recorded
    // reset carries the programmatic attribute, and only when the handle's previous operation was a step launch that released
    // its epoch (ovl_chain): a predecessor that does not trigger lets the launch start once its blocks have exited, before its
    // writes need be visible, and the epochs cover only what step launches wrote.  Everything that step reads is the
    // handle's own state; other work on the stream between two steps may read their outputs but writes nothing it
    // reads.  Steps fed actions from outside (step, step_obs), fused resets (caller's weights) and every step after
    // another call on the handle wait for their predecessor in full.  A launch being captured into a graph takes no
    // part: its epoch would be released only when the graph runs.
    bool pdl = false;
    if (S::OVL && (MODE & MODE_STEP) && !(MODE & MODE_HOST) && h->launch_overlap) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cs) != cudaSuccess) {
            cudaGetLastError();
            cs = cudaStreamCaptureStatusActive;
        }
        if (cs == cudaStreamCaptureStatusNone) {
            pdl = (MODE & MODE_POLICY) && !(MODE & MODE_FROM_RESET) && h->ovl_chain;
            Q.done_ep = h->done_ep;
            Q.ovl_err = h->ovl_err_d;
            Q.wait_ep = pdl ? h->ep : 0;
            Q.ep = h->ep + 1;
        }
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(S::WARPS * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[2];
    cfg.attrs = at;
    if (h->window_bytes && (MODE & MODE_STEP)) {
        cudaLaunchAttribute& a = at[cfg.numAttrs++];
        a.id = cudaLaunchAttributeAccessPolicyWindow;
        a.val.accessPolicyWindow.base_ptr = h->slab;
        a.val.accessPolicyWindow.num_bytes = h->window_bytes;
        a.val.accessPolicyWindow.hitRatio = 1.0f;
        a.val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        a.val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    if (pdl) {
        cudaLaunchAttribute& a = at[cfg.numAttrs++];
        a.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        a.val.programmaticStreamSerializationAllowed = 1;
    }
    h->ovl_chain = false;
    CK(cudaLaunchKernelEx(&cfg, env_kernel_s<S, MODE, OutT>, Q), "env_kernel_s launch");
    h->launches++;
    CK(cudaGetLastError(), "env_kernel_s launch");
    if (Q.ep) {  // only a launch that was issued releases its epoch
        h->ep = Q.ep;
        h->ovl_chain = true;
    }
    return MTFJSP_OK;
}

// Sizes with a specialised kernel: the benchmark configurations of BASELINE.json and the size list of the reference's
// instance generator (instance/generate_allsize_mofjsp_dataset.py:429); everything else (and the first reset) runs the
// generic one-warp-per-env kernel.  X(J, M, lanes per env, warps per block): lanes >= max(J, M), 32 when N > 128; warps per block = what
// keeps the most envs resident (shared memory per env is the limiter).
#define MTFJSP_SPEC_SIZES(X) \
    X(6, 6, 8, 4, false) X(10, 6, 16, 1, false) X(20, 6, 32, 1, false) X(10, 10, 16, 1, false) X(15, 10, 32, 1, true) \
    X(20, 10, 32, 1, true) X(30, 20, 32, 1, true)

static bool has_spec(int J, int M) {
#define X(JJ, MM, GG, WW, CC) if (J == JJ && M == MM) return true;
    MTFJSP_SPEC_SIZES(X)
#undef X
    return false;
}

template <int MODE, typename OutT>
static int launch_env_auto(mtfjsp_env* h, const Params& P, cudaStream_t s) {
    if (!(MODE & MODE_RESET) && !h->force_generic) {
        const int J = h->L.J, M = h->L.M;
#define X(JJ, MM, GG, WW, CC) if (J == JJ && M == MM) return launch_spec<Spec<JJ, MM, GG, WW, CC>, MODE, OutT>(h, P, s);
        MTFJSP_SPEC_SIZES(X)
#undef X
    }
    return launch_env<MODE & ~MODE_HOST, OutT>(h, P, s);
}

// random-rollout step in one launch (policy + candidate-machine features + step + observation): sizes with a
// specialised kernel only.  Returns 1 if launched, 0 if the size has none (caller runs the separate kernels), <0 on error.
template <typename OutT>
static int launch_random_fused(mtfjsp_env* h, const Params& P, cudaStream_t s) {
    if (h->force_generic || !h->fuse_policy) return 0;
    constexpr int MD = MODE_STEP | MODE_OBS | MODE_POLICY;
    const int J = h->L.J, M = h->L.M;
#define X(JJ, MM, GG, WW, CC)                                                    \
    if (J == JJ && M == MM) {                                                    \
        const int rc = launch_spec<Spec<JJ, MM, GG, WW, CC>, MD, OutT>(h, P, s); \
        return rc == MTFJSP_OK ? 1 : rc;                                         \
    }
    MTFJSP_SPEC_SIZES(X)
#undef X
    return 0;
}

// pre-step dispatch: returns 1 if a size-templated kernel was launched, 0 if the size has none, <0 on error
template <bool POLICY>
static int launch_prestep(mtfjsp_env* h, uint64_t seed, uint64_t env_offset, const uint8_t* jm, int32_t* op,
                          int32_t* mach, void* out, uint8_t* mmask, int dtype, cudaStream_t s) {
    if (h->force_generic) return 0;
    const Layout& L = h->L;
    const unsigned blocks = (unsigned)((L.B + 127) / 128);
#define PRESTEP(MM)                                                                                                  \
    if (L.M == MM) {                                                                                                 \
        if (dtype == MTFJSP_F64)                                                                                     \
            prestep_kernel<MM, double, POLICY><<<blocks, 128, 0, s>>>(L, h->t, h->p, h->xs, h->si, h->edge_id, jm,    \
                                                                     h->cand, seed, env_offset, op, mach,            \
                                                                     (double*)out, mmask);                           \
        else                                                                                                         \
            prestep_kernel<MM, float, POLICY><<<blocks, 128, 0, s>>>(L, h->t, h->p, h->xs, h->si, h->edge_id, jm,     \
                                                                    h->cand, seed, env_offset, op, mach, (float*)out, \
                                                                    mmask);                                          \
        h->launches++;                                                                                               \
        CK(cudaGetLastError(), "prestep_kernel");                                                                    \
        return 1;                                                                                                    \
    }
    PRESTEP(6)
    PRESTEP(10)
    PRESTEP(20)
#undef PRESTEP
    return 0;
}

static int fill_obs(mtfjsp_env* h, Params& P, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src,
                    uint8_t* job_mask, int32_t* candidate, int mask_mode, int dtype) {
    if (dtype != MTFJSP_F32 && dtype != MTFJSP_F64) return fail(MTFJSP_E_ARG, "dtype must be MTFJSP_F32 or MTFJSP_F64");
    if (mask_mode != MTFJSP_MASK_ESA && mask_mode != MTFJSP_MASK_FINISHED) return fail(MTFJSP_E_ARG, "bad mask_mode");
    if ((adj_w == nullptr) != (adj_src == nullptr)) return fail(MTFJSP_E_ARG, "adj_w and adj_src go together");
    P.tfea = task_fea; P.mfea = mach_fea; P.adj_w = adj_w; P.adj_src = adj_src; P.jmask = job_mask; P.cand = candidate;
    P.mask_mode = mask_mode;
    (void)h;
    return MTFJSP_OK;
}

// Incremental observation bookkeeping.  A fused step may rewrite only the changed rows iff the caller's output buffers
// already hold the observation of the current state: the same four pointers and dtype received a full observation
// (mtfjsp_obs, or a fused step that wrote everything) since the last reset / load / observation-less step, and every
// step since went through them.  obs_inc_now() answers that before a whole-batch step, obs_mark() records it after.
static int obs_inc_now(const mtfjsp_env* h, const void* tfea, const void* mfea, const void* adj_w, const void* adj_src,
                       int dtype) {
    return h->obs_inc_enabled && h->obs_synced && h->obs_dtype == dtype && h->obs_ptrs[0] == tfea &&
           h->obs_ptrs[1] == mfea && h->obs_ptrs[2] == adj_w && h->obs_ptrs[3] == adj_src;
}
static void obs_mark(mtfjsp_env* h, const void* tfea, const void* mfea, const void* adj_w, const void* adj_src, int dtype) {
    h->obs_synced = true;
    h->obs_dtype = dtype;
    h->obs_ptrs[0] = tfea; h->obs_ptrs[1] = mfea; h->obs_ptrs[2] = adj_w; h->obs_ptrs[3] = adj_src;
}

// fused step + observation over the whole batch
static int launch_step_obs(mtfjsp_env* h, const int32_t* op, const int32_t* mach, double* reward5, double* scaled4,
                           uint8_t* done, uint8_t* invalid, double* info6, void* task_fea, void* mach_fea, float* adj_w,
                           int16_t* adj_src, uint8_t* job_mask, int32_t* candidate, int mask_mode, int dtype,
                           cudaStream_t s, const int2* act2 = nullptr, unsigned char* rec = nullptr, int obs_inc = 0) {
    Params P = make_params(h);
    P.op = op; P.mach = mach; P.reward5 = reward5; P.scaled4 = scaled4; P.done = done; P.invalid = invalid;
    P.info6 = info6; P.act2 = act2; P.rec = rec; P.rec_stride = h->rec_stride;
    P.obs_inc = obs_inc;
    int rc = fill_obs(h, P, task_fea, mach_fea, adj_w, adj_src, job_mask, candidate, mask_mode, dtype);
    if (rc) return rc;
    if (rec || info6)  // host-step calls: the variant that stages these outputs and writes them as whole-warp runs
        return dtype == MTFJSP_F64 ? launch_env_auto<MODE_STEP | MODE_OBS | MODE_HOST, double>(h, P, s)
                                   : launch_env_auto<MODE_STEP | MODE_OBS | MODE_HOST, float>(h, P, s);
    return dtype == MTFJSP_F64 ? launch_env_auto<MODE_STEP | MODE_OBS, double>(h, P, s)
                               : launch_env_auto<MODE_STEP | MODE_OBS, float>(h, P, s);
}

extern "C" {

const char* mtfjsp_last_error(void) { return g_err; }
const char* mtfjsp_version(void) { return "mtfjsp-b200 0.1 (sm_100a)"; }

int mtfjsp_create(mtfjsp_env** out, int B, int J, int M, int E, int left_shift, int device) {
    if (!out) return fail(MTFJSP_E_ARG, "null handle pointer");
    *out = nullptr;
    if (B < 1 || J < 1 || M < 2 || M > 64 || E < 1 || (long long)J * M > 4096)
        return fail(MTFJSP_E_ARG, "size out of range (need B>=1, J>=1, 2<=M<=64, J*M<=4096, E>=1, and one env's state "
                                  "within one block's shared memory: J<=48 at M=64, J<=109 at M=32, J<=1678 at M=2)");
    CK(cudaSetDevice(device), "cudaSetDevice");
    mtfjsp_env* h = new (std::nothrow) mtfjsp_env();
    if (!h) return fail(MTFJSP_E_ARG, "out of host memory");
    memset(h, 0, sizeof *h);
    Layout& L = h->L;
    const int N = J * M;
    L.B = B; L.J = J; L.M = M; L.N = N; L.E = E; L.left_shift = left_shift ? 1 : 0;
    L.o_st = 0; L.o_ft = N; L.o_dur = 2 * N; L.o_psel = 3 * N; L.o_scal = 4 * N; L.o_macc = 4 * N + 4;
    h->pw.nleaves = 0; h->pw.nprog = 0;
    build_plan_rec(0, N, h->pw);
    L.o_w = L.o_macc + 3 * M; L.o_eacc = L.o_w + 3; L.o_eleaf = L.o_eacc + 8 * h->pw.nleaves;
    L.o_ipre = L.o_eleaf + (h->pw.nleaves > 1 ? h->pw.nleaves : 0);  // a single leaf's result is the total: not cached
    L.nich = N > 128 ? (N + 31) / 32 : 0;
    L.o_sc = L.o_ipre + L.nich;
    L.sd_stride = align_up(L.o_sc + 13, 2);
    L.o_mach = 0; L.o_ord = N; L.o_rpred = 2 * N; L.o_cnt = 3 * N; L.o_misc = 3 * N + M;
    L.o_nxt = L.o_misc + 3;
    L.si_stride = align_up(L.o_nxt + J, 8);
    L.o_mind = 0; L.o_minpt = N; L.o_tt = 2 * N;
    L.xs_stride = align_up(2 * N + M * M, 2);
    int off = 0;
    L.sm_sd = off; off += L.sd_stride * 8;
    L.sm_xs = off; off += L.xs_stride * 8;
    L.sm_pt = off; off += align_up(N, 2) * 8;
    L.sm_v = off; off += align_up(J, 2) * 8;
    L.sm_leaf = off; off += (MAX_LEAVES + 32) * 8;
    L.sm_si = off; off += L.si_stride * 2;
    L.sm_off = off; off += align_up(M, 4) * 4;
    L.sm_nxt = off; off += align_up(J, 8) * 2;
    L.sm_tail = off; off += align_up(M, 8) * 2;
    L.smem_per_warp = align_up(off, 16);
    int wpb = 8;
    while (wpb > 1 && (size_t)wpb * L.smem_per_warp > 200 * 1024) wpb >>= 1;
    if ((size_t)wpb * L.smem_per_warp > 227 * 1024) {  // about 62 * N + 8 * M * M bytes per env (include/mtfjsp.h)
        delete h;
        return fail(MTFJSP_E_ARG, "instance too large: one env's state exceeds one block's shared memory (227 KB); "
                                  "the largest J is 48 at M=64, 109 at M=32, 1678 at M=2");
    }
    L.warps_per_block = wpb;
    h->device = device;
    {
        const char* fg = getenv("MTFJSP_FORCE_GENERIC");  // test hook: run the generic kernel on every size
        h->force_generic = fg && fg[0] == '1';
        // test hook (1 | 2); default: from 16,384 envs up (below that the explicit copy is as fast)
        h->host_act_in_place = getenv("MTFJSP_HOST_ZEROCOPY") ? atoi(getenv("MTFJSP_HOST_ZEROCOPY")) >= 2 : B >= 16384;
        h->fuse_policy = getenv("MTFJSP_FUSE_POLICY") ? atoi(getenv("MTFJSP_FUSE_POLICY")) : 1;
        h->obs_inc_allowed = !(getenv("MTFJSP_OBS_INCREMENTAL") && atoi(getenv("MTFJSP_OBS_INCREMENTAL")) == 0);  // test hook
        h->fused_reset = getenv("MTFJSP_FUSED_RESET") ? atoi(getenv("MTFJSP_FUSED_RESET")) : 1;
        h->launch_overlap = getenv("MTFJSP_LAUNCH_OVERLAP") ? atoi(getenv("MTFJSP_LAUNCH_OVERLAP")) : 1;
    }
    h->cfgw[0] = 0.4; h->cfgw[1] = 0.4; h->cfgw[2] = 0.2; h->divisor = 1.0; h->gamma = 0.99;
    size_t Bs = (size_t)B;
#define ALLOC(ptr, bytes)                                                      \
    do {                                                                       \
        cudaError_t e_ = cudaMalloc((void**)&(ptr), (bytes));                  \
        if (e_ != cudaSuccess) { mtfjsp_destroy(h); return fail(MTFJSP_E_CUDA, "cudaMalloc", e_); } \
        cudaMemset((ptr), 0, (bytes));                                         \
    } while (0)
    ALLOC(h->sd, Bs * L.sd_stride * 8);
    {
        auto up = [](size_t x) { return (x + 255) / 256 * 256; };
        const size_t b_si = up(Bs * L.si_stride * 2), b_jm = up(Bs * J), b_cd = up(Bs * J * 4), b_xs = up(Bs * L.xs_stride * 8);
        h->slab_bytes = b_si + 2 * b_jm + b_cd + b_xs;
        ALLOC(h->slab, h->slab_bytes);
        h->jm_fin = h->slab;
        h->jm_esa = h->slab + b_jm;
        h->cand = reinterpret_cast<int32_t*>(h->slab + 2 * b_jm);
        h->si = reinterpret_cast<int16_t*>(h->slab + 2 * b_jm + b_cd);
        h->xs = reinterpret_cast<double*>(h->slab + 2 * b_jm + b_cd + b_si);  // static tables (transport table, min durations)
        h->window_bytes = 0;
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
            size_t want = h->slab_bytes - b_xs;  // the window leaves out the static tables
            if (want > (size_t)prop.accessPolicyMaxWindowSize) want = (size_t)prop.accessPolicyMaxWindowSize;
            size_t carve = want < (size_t)prop.persistingL2CacheMaxSize ? want : (size_t)prop.persistingL2CacheMaxSize;
            size_t cur = 0;
            cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize);
            if (cur < carve) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
            h->window_bytes = want;
        }
        cudaGetLastError();
    }
    ALLOC(h->t, Bs * N * M * 8);
    ALLOC(h->p, Bs * N * M * 8);
    ALLOC(h->edge_id, Bs * M);
    ALLOC(h->a_op, Bs * 4);
    ALLOC(h->a_mach, Bs * 4);
    ALLOC(h->r5, Bs * 5 * 8);
    ALLOC(h->s4, Bs * 4 * 8);
    ALLOC(h->info6, Bs * 6 * 8);
    h->rec_stride = rec_bytes(J);
    ALLOC(h->act2, Bs * 8);
    ALLOC(h->rec, Bs * h->rec_stride);
    ALLOC(h->dn, Bs);
    ALLOC(h->inv, Bs);
    ALLOC(h->tmp_adj_w, Bs * N * 2 * 4);
    ALLOC(h->tmp_adj_src, Bs * N * 2);
    ALLOC(h->sd0, Bs * L.sd_stride * 8);
    ALLOC(h->si0, Bs * L.si_stride * 2);
    ALLOC(h->done_ep, Bs * sizeof(unsigned long long));  // at most one entry per env
#undef ALLOC
    {
        cudaError_t e_ = cudaHostAlloc((void**)&h->ovl_err, sizeof(unsigned), cudaHostAllocMapped);
        if (e_ == cudaSuccess) { *h->ovl_err = 0; e_ = cudaHostGetDevicePointer((void**)&h->ovl_err_d, h->ovl_err, 0); }
        if (e_ != cudaSuccess) { mtfjsp_destroy(h); return fail(MTFJSP_E_CUDA, "cudaHostAlloc", e_); }
    }
    *out = h;
    return MTFJSP_OK;
}

int mtfjsp_destroy(mtfjsp_env* h) {
    if (!h) return MTFJSP_OK;
    cudaSetDevice(h->device);
    void* ptrs[] = {h->sd, h->slab, h->t, h->p, h->edge_id, h->a_op, h->a_mach,
                    h->r5, h->s4, h->info6, h->dn, h->inv, h->tmp_adj_w, h->tmp_adj_src, h->act2, h->rec, h->sd0, h->si0, h->done_ep};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    if (h->ovl_err) cudaFreeHost(h->ovl_err);
    delete h;
    return MTFJSP_OK;
}

int mtfjsp_set_params(mtfjsp_env* h, double w_mk, double w_ec, double w_tt, double scaling_divisor, double gamma) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    if (scaling_divisor == 0.0) return fail(MTFJSP_E_ARG, "scaling_divisor must be non-zero");
    h->cfgw[0] = w_mk; h->cfgw[1] = w_ec; h->cfgw[2] = w_tt; h->divisor = scaling_divisor; h->gamma = gamma;
    return MTFJSP_OK;
}

int mtfjsp_set_obs_incremental(mtfjsp_env* h, int on) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    h->obs_inc_enabled = on != 0 && h->obs_inc_allowed;
    h->obs_synced = false;
    return MTFJSP_OK;
}

int mtfjsp_load(mtfjsp_env* h, const double* t, const double* p, const double* tt, const int32_t* edge, int W,
                void* stream) {
    if (!h || !t || !p || !tt || !edge || W < 1) return fail(MTFJSP_E_ARG, "mtfjsp_load: bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = enter(h, s);
    if (rc) return rc;
    const Layout& L = h->L;
    size_t n = (size_t)L.B * L.N * L.M * 8;
    CK(cudaMemcpyAsync(h->t, t, n, cudaMemcpyDeviceToDevice, s), "copy t");
    CK(cudaMemcpyAsync(h->p, p, n, cudaMemcpyDeviceToDevice, s), "copy p");
    size_t total = (size_t)L.B * (size_t)(L.N > L.M * L.M ? L.N : L.M * L.M);
    load_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(L, h->t, h->p, tt, edge, W, h->xs, h->edge_id);
    h->launches++;
    CK(cudaGetLastError(), "load_kernel");
    h->loaded = true;
    h->reset_done = false;
    h->obs_synced = false;
    h->reset_snap = false;
    return MTFJSP_OK;
}

int mtfjsp_scaler_init(mtfjsp_env* h, void* stream) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    size_t n = (size_t)h->L.B * 13;
    scaler_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->L, h->sd, 1);
    h->launches++;
    CK(cudaGetLastError(), "scaler_kernel");
    return MTFJSP_OK;
}

int mtfjsp_scaler_reset(mtfjsp_env* h, void* stream) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    if (h->pend_reset) {  // performed together with the recorded reset
        h->pend_scaler = true;
        return MTFJSP_OK;
    }
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    size_t n = (size_t)h->L.B * 4;
    scaler_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->L, h->sd, 0);
    h->launches++;
    CK(cudaGetLastError(), "scaler_kernel");
    return MTFJSP_OK;
}

int mtfjsp_reset(mtfjsp_env* h, const double* weights, void* stream) {
    if (!h || !weights) return fail(MTFJSP_E_ARG, "mtfjsp_reset: bad argument");
    if (!h->loaded) return fail(MTFJSP_E_STATE, "mtfjsp_reset before mtfjsp_load");
    cudaStream_t s = (cudaStream_t)stream;
    const Layout& L = h->L;
    h->obs_synced = false;
    if (h->reset_snap) {  // recorded; a later reset replaces the weights, a pending scaler reset stays
        h->pend_reset = true;
        h->pend_w = weights;
        return h->fused_reset ? MTFJSP_OK : enter(h, s);
    }
    CK(cudaSetDevice(h->device), "cudaSetDevice");
    Params P = make_params(h);
    P.weights = weights;
    int rc = launch_env<MODE_RESET, double>(h, P, s);
    if (rc != MTFJSP_OK) return rc;
    h->reset_done = true;
    CK(cudaMemcpyAsync(h->sd0, h->sd, (size_t)L.B * L.sd_stride * 8, cudaMemcpyDeviceToDevice, s), "snapshot sd");
    CK(cudaMemcpyAsync(h->si0, h->si, (size_t)L.B * L.si_stride * 2, cudaMemcpyDeviceToDevice, s), "snapshot si");
    h->reset_snap = true;
    return MTFJSP_OK;
}


int mtfjsp_step(mtfjsp_env* h, const int32_t* op, const int32_t* mach, double* reward5, double* scaled4,
                uint8_t* done, uint8_t* invalid, void* stream) {
    if (!h || !op || !mach) return fail(MTFJSP_E_ARG, "mtfjsp_step: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_step before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream, true);
    if (rc) return rc;
    Params P = make_params(h);
    P.op = op; P.mach = mach; P.reward5 = reward5; P.scaled4 = scaled4; P.done = done; P.invalid = invalid;
    h->obs_synced = false;  // the state moves on without any observation buffer following it
    return launch_env_auto<MODE_STEP, double>(h, P, (cudaStream_t)stream);
}

int mtfjsp_obs(mtfjsp_env* h, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src, uint8_t* job_mask,
               int32_t* candidate, int mask_mode, int dtype, void* stream) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_obs before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    Params P = make_params(h);
    rc = fill_obs(h, P, task_fea, mach_fea, adj_w, adj_src, job_mask, candidate, mask_mode, dtype);
    if (rc) return rc;
    rc = dtype == MTFJSP_F64 ? launch_env_auto<MODE_OBS, double>(h, P, (cudaStream_t)stream)
                             : launch_env_auto<MODE_OBS, float>(h, P, (cudaStream_t)stream);
    // a full observation into a complete buffer set makes that set the mirror of the state -- unless another set already
    // is (a side view such as mtfjsp_dense_adj must not break the main buffers' chain)
    if (rc == MTFJSP_OK && task_fea && mach_fea && adj_w && !h->obs_synced) obs_mark(h, task_fea, mach_fea, adj_w, adj_src, dtype);
    return rc;
}

int mtfjsp_step_obs(mtfjsp_env* h, const int32_t* op, const int32_t* mach, double* reward5, double* scaled4,
                    uint8_t* done, uint8_t* invalid, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src,
                    uint8_t* job_mask, int32_t* candidate, int mask_mode, int dtype, void* stream) {
    if (!h || !op || !mach) return fail(MTFJSP_E_ARG, "mtfjsp_step_obs: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_step_obs before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream, true);
    if (rc) return rc;
    const int inc = obs_inc_now(h, task_fea, mach_fea, adj_w, adj_src, dtype);
    rc = launch_step_obs(h, op, mach, reward5, scaled4, done, invalid, nullptr, task_fea, mach_fea, adj_w, adj_src,
                         job_mask, candidate, mask_mode, dtype, (cudaStream_t)stream, nullptr, nullptr, inc);
    if (rc == MTFJSP_OK) obs_mark(h, task_fea, mach_fea, adj_w, adj_src, dtype);
    return rc;
}

int mtfjsp_mfea1(mtfjsp_env* h, const int32_t* op, void* mfea1, uint8_t* mach_mask, int dtype, void* stream) {
    if (!h || !op || !mfea1) return fail(MTFJSP_E_ARG, "mtfjsp_mfea1: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_mfea1 before mtfjsp_reset");
    const Layout& L = h->L;
    cudaStream_t s = (cudaStream_t)stream;
    {
        int rc = enter(h, s);
        if (rc) return rc;
    }
    if (dtype != MTFJSP_F32 && dtype != MTFJSP_F64) return fail(MTFJSP_E_ARG, "dtype must be MTFJSP_F32 or MTFJSP_F64");
    {
        int rc = launch_prestep<false>(h, 0, 0, nullptr, const_cast<int32_t*>(op), nullptr, mfea1, mach_mask, dtype, s);
        if (rc != 0) return rc < 0 ? rc : MTFJSP_OK;
    }
    unsigned blocks = (unsigned)((L.B + 127) / 128);
    if (dtype == MTFJSP_F64)
        mfea1_kernel<double><<<blocks, 128, 0, s>>>(L, h->t, h->p, h->xs, h->si, h->edge_id, op, (double*)mfea1, mach_mask);
    else if (dtype == MTFJSP_F32)
        mfea1_kernel<float><<<blocks, 128, 0, s>>>(L, h->t, h->p, h->xs, h->si, h->edge_id, op, (float*)mfea1, mach_mask);
    else
        return fail(MTFJSP_E_ARG, "dtype must be MTFJSP_F32 or MTFJSP_F64");
    h->launches++;
    CK(cudaGetLastError(), "mfea1_kernel");
    return MTFJSP_OK;
}

int mtfjsp_dense_adj(mtfjsp_env* h, void* adj, int dtype, void* stream) {
    if (!h || !adj) return fail(MTFJSP_E_ARG, "mtfjsp_dense_adj: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_dense_adj before mtfjsp_reset");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = enter(h, s);
    if (rc) return rc;
    rc = mtfjsp_obs(h, nullptr, nullptr, h->tmp_adj_w, h->tmp_adj_src, nullptr, nullptr, MTFJSP_MASK_ESA, MTFJSP_F32, stream);
    if (rc) return rc;
    if (dtype == MTFJSP_F64) dense_adj_kernel<double><<<h->L.B, 256, 0, s>>>(h->L, h->tmp_adj_w, h->tmp_adj_src, (double*)adj);
    else if (dtype == MTFJSP_F32) dense_adj_kernel<float><<<h->L.B, 256, 0, s>>>(h->L, h->tmp_adj_w, h->tmp_adj_src, (float*)adj);
    else return fail(MTFJSP_E_ARG, "dtype must be MTFJSP_F32 or MTFJSP_F64");
    h->launches++;
    CK(cudaGetLastError(), "dense_adj_kernel");
    return MTFJSP_OK;
}

int mtfjsp_raw_adj(mtfjsp_env* h, int32_t* adj, void* stream) {
    if (!h || !adj) return fail(MTFJSP_E_ARG, "mtfjsp_raw_adj: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_raw_adj before mtfjsp_reset");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = enter(h, s);
    if (rc) return rc;
    const Layout& L = h->L;
    CK(cudaMemsetAsync(adj, 0, (size_t)L.B * L.N * L.N * sizeof(int32_t), s), "cudaMemsetAsync");
    const size_t n = (size_t)L.B * L.N;
    raw_adj_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(L, h->sd, h->si, h->xs, adj);
    h->launches++;
    CK(cudaGetLastError(), "raw_adj_kernel");
    return MTFJSP_OK;
}

int mtfjsp_generate_instances(int B, int J, int M, int E, uint64_t seed, uint64_t env_offset, double* t, double* p, double* tt,
                              int32_t* edge, int W, void* stream) {
    if (B < 1 || J < 1 || M < 2 || M > 64 || E < 1 || E > M || !t || !p || !tt || !edge)
        return fail(MTFJSP_E_ARG, "mtfjsp_generate_instances: bad argument");
    const int avg = M / E, wmin = M - avg * (E - 1);
    if (W < wmin || W < avg || (long long)E * W > (long long)J * M || (long long)M * M > (long long)J * M * 64)
        return fail(MTFJSP_E_ARG, "mtfjsp_generate_instances: edge table width too small (need W >= largest group) or sizes out of range");
    if ((long long)M * M > (long long)J * M) return fail(MTFJSP_E_ARG, "mtfjsp_generate_instances: needs J >= M");
    const size_t n = (size_t)B * J * M;
    instance_gen_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(B, J, M, E, W, seed, env_offset, t, p, tt, edge);
    CK(cudaGetLastError(), "instance_gen_kernel");
    return MTFJSP_OK;
}

int mtfjsp_costs(mtfjsp_env* h, double* cost4, double* total_e1, void* stream) {
    if (!h || (!cost4 && !total_e1)) return fail(MTFJSP_E_ARG, "mtfjsp_costs: bad argument");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    costs_kernel<<<(h->L.B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->L, h->sd, cost4, total_e1);
    h->launches++;
    CK(cudaGetLastError(), "costs_kernel");
    return MTFJSP_OK;
}

int mtfjsp_export_state(mtfjsp_env* h, int32_t* mach, double* st, double* ft, int32_t* routes, void* stream) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = enter(h, s);
    if (rc) return rc;
    const Layout& L = h->L;
    if (routes) {
        size_t n = (size_t)L.B * L.M * L.N;
        fill_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(routes, n, -1);
        h->launches++;
    }
    size_t n = (size_t)L.B * L.N;
    export_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(L, h->sd, h->si, mach, st, ft, routes);
    h->launches++;
    CK(cudaGetLastError(), "export_kernel");
    return MTFJSP_OK;
}

int mtfjsp_export_scaler(mtfjsp_env* h, double* R, double* mean, double* S, int64_t* n, void* stream) {
    if (!h || !R || !mean || !S || !n) return fail(MTFJSP_E_ARG, "mtfjsp_export_scaler: bad argument");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    export_scaler_kernel<<<(h->L.B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->L, h->sd, R, mean, S, n);
    h->launches++;
    CK(cudaGetLastError(), "export_scaler_kernel");
    return MTFJSP_OK;
}

int mtfjsp_gather(mtfjsp_env* dst, const mtfjsp_env* src, const int32_t* idx, void* stream) {
    if (!dst || !src || !idx) return fail(MTFJSP_E_ARG, "mtfjsp_gather: bad argument");
    if (dst == src) return fail(MTFJSP_E_ARG, "mtfjsp_gather: src and dst are the same handle (no in-place gather)");
    if (dst->device != src->device) return fail(MTFJSP_E_ARG, "mtfjsp_gather: src and dst live on different devices");
    const Layout &Ld = dst->L, &Ls = src->L;
    if (Ld.J != Ls.J || Ld.M != Ls.M || Ld.E != Ls.E || Ld.left_shift != Ls.left_shift)
        return fail(MTFJSP_E_ARG, "mtfjsp_gather: src and dst differ in (J, M, E, left_shift)");
    if (dst->cfgw[0] != src->cfgw[0] || dst->cfgw[1] != src->cfgw[1] || dst->cfgw[2] != src->cfgw[2] ||
        dst->divisor != src->divisor || dst->gamma != src->gamma)
        return fail(MTFJSP_E_ARG, "mtfjsp_gather: src and dst differ in mtfjsp_set_params (weights, divisor, gamma)");
    if (!src->loaded) return fail(MTFJSP_E_STATE, "mtfjsp_gather from a handle that was never loaded");
    cudaStream_t s = (cudaStream_t)stream;
    // a non-step call on both handles: recorded resets run now (src's belongs to the copied state; dst's next step would
    // otherwise perform its own on the copy), and the next step of either waits for the copy in full
    mtfjsp_env* hs = const_cast<mtfjsp_env*>(src);
    int rc = enter(hs, s);
    if (rc) return rc;
    rc = enter(dst, s);
    if (rc) return rc;
    GatherArgs A;
    memset(&A, 0, sizeof A);
    A.L = Ld; A.src_B = Ls.B; A.idx = idx;
    A.sd = hs->sd; A.sd0 = hs->sd0; A.xs = hs->xs; A.t = hs->t; A.p = hs->p; A.si = hs->si; A.si0 = hs->si0;
    A.edge_id = hs->edge_id; A.jm_fin = hs->jm_fin; A.jm_esa = hs->jm_esa; A.dn = hs->dn; A.inv = hs->inv; A.cand = hs->cand;
    A.d_sd = dst->sd; A.d_sd0 = dst->sd0; A.d_xs = dst->xs; A.d_t = dst->t; A.d_p = dst->p; A.d_si = dst->si; A.d_si0 = dst->si0;
    A.d_edge_id = dst->edge_id; A.d_jm_fin = dst->jm_fin; A.d_jm_esa = dst->jm_esa; A.d_dn = dst->dn; A.d_inv = dst->inv;
    A.d_cand = dst->cand;
    gather_kernel<<<Ld.B, 128, 0, s>>>(A);
    dst->launches++;
    CK(cudaGetLastError(), "gather_kernel");
    dst->loaded = true;
    dst->reset_done = hs->reset_done;
    dst->reset_snap = hs->reset_snap;
    dst->obs_synced = false;  // the caller's observation buffers no longer mirror dst's state
    return MTFJSP_OK;
}

int mtfjsp_peek(mtfjsp_env* h, const int32_t* op, const int32_t* mach, int K, double* reward5, uint8_t* invalid,
                void* stream) {
    if (!h || !op || !mach || K < 1) return fail(MTFJSP_E_ARG, "mtfjsp_peek: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_peek before mtfjsp_reset");
    const Layout& L = h->L;
    const int warps = 4;
    const size_t smem = (size_t)peek_smem(L, h->pw.nleaves, warps).total;
    if (smem > 227 * 1024) return fail(MTFJSP_E_ARG, "mtfjsp_peek: one env's records exceed one block's shared memory");
    cudaStream_t s = (cudaStream_t)stream;
    // a non-step call: a recorded reset runs now, and the next step waits for the peek in full
    int rc = enter(h, s);
    if (rc) return rc;
    static thread_local int configured_dev = -1;
    static thread_local size_t configured_smem = 0;
    if (smem > 48 * 1024 && (configured_dev != h->device || configured_smem < smem)) {
        CK(cudaFuncSetAttribute(peek_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute");
        configured_dev = h->device;
        configured_smem = smem;
    }
    PeekArgs A;
    memset(&A, 0, sizeof A);
    A.L = L; A.pw = h->pw;
    A.sd = h->sd; A.xs = h->xs; A.t = h->t; A.p = h->p; A.si = h->si;
    A.op = op; A.mach = mach; A.K = K;
    A.cfgw[0] = h->cfgw[0]; A.cfgw[1] = h->cfgw[1]; A.cfgw[2] = h->cfgw[2]; A.divisor = h->divisor;
    A.reward5 = reward5; A.invalid = invalid;
    peek_kernel<<<L.B, warps * 32, smem, s>>>(A);
    h->launches++;
    CK(cudaGetLastError(), "peek_kernel");
    return MTFJSP_OK;
}

int mtfjsp_replay(mtfjsp_env* h, const int32_t* src, int R, const int32_t* actions, int T, double* cost4, double* return5,
                  int32_t* first_invalid, void* stream) {
    if (!h || !src || !actions || R < 1 || T < 1 || T > h->L.N) return fail(MTFJSP_E_ARG, "mtfjsp_replay: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_replay before mtfjsp_reset");
    const Layout& L = h->L;
    cudaStream_t s = (cudaStream_t)stream;
    // a non-step call: a recorded reset runs now, and the next step waits for the replay in full
    int rc = enter(h, s);
    if (rc) return rc;
    const size_t smem = (size_t)L.smem_per_warp * L.warps_per_block;
    static thread_local int configured_dev = -1;
    static thread_local size_t configured_smem = 0;
    if (configured_dev != h->device || configured_smem < smem) {
        CK(cudaFuncSetAttribute(replay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute");
        configured_dev = h->device;
        configured_smem = smem;
    }
    ReplayArgs A;
    memset(&A, 0, sizeof A);
    A.L = L; A.pw = h->pw;
    A.sd0 = h->sd0; A.xs = h->xs; A.t = h->t; A.p = h->p; A.si0 = h->si0;
    A.src = src; A.actions = actions; A.R = R; A.T = T;
    A.cfgw[0] = h->cfgw[0]; A.cfgw[1] = h->cfgw[1]; A.cfgw[2] = h->cfgw[2]; A.divisor = h->divisor;
    A.cost4 = cost4; A.return5 = return5; A.first_invalid = first_invalid;
    const unsigned blocks = (unsigned)((R + L.warps_per_block - 1) / L.warps_per_block);
    replay_kernel<<<blocks, L.warps_per_block * 32, smem, s>>>(A);
    h->launches++;
    CK(cudaGetLastError(), "replay_kernel");
    return MTFJSP_OK;
}

int mtfjsp_policy_random(mtfjsp_env* h, uint64_t seed, uint64_t env_offset, int mask_mode, int32_t* op,
                         int32_t* mach, void* stream) {
    if (!h || !op || !mach) return fail(MTFJSP_E_ARG, "mtfjsp_policy_random: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_policy_random before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    const uint8_t* jm = mask_mode == MTFJSP_MASK_ESA ? h->jm_esa : h->jm_fin;
    policy_kernel<<<(h->L.B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->L, h->t, h->si, jm, h->cand, seed, env_offset, op, mach);
    h->launches++;
    CK(cudaGetLastError(), "policy_kernel");
    return MTFJSP_OK;
}

int mtfjsp_random_step(mtfjsp_env* h, uint64_t seed, uint64_t env_offset, int32_t* op, int32_t* mach, void* mfea1,
                       uint8_t* mach_mask, double* reward5, double* scaled4, uint8_t* done, uint8_t* invalid,
                       void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src, uint8_t* job_mask,
                       int32_t* candidate, int mask_mode, int dtype, void* stream) {
    if (!h) return fail(MTFJSP_E_ARG, "null handle");
    int32_t* o = op ? op : h->a_op;
    int32_t* mc = mach ? mach : h->a_mach;
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_random_step before mtfjsp_reset");
    if (dtype != MTFJSP_F32 && dtype != MTFJSP_F64) return fail(MTFJSP_E_ARG, "dtype must be MTFJSP_F32 or MTFJSP_F64");
    int rc = enter(h, (cudaStream_t)stream, true);
    if (rc) return rc;
    {
        Params P = make_params(h);
        P.reward5 = reward5; P.scaled4 = scaled4; P.done = done; P.invalid = invalid;
        P.seed = seed; P.env_offset = env_offset; P.edge_id = h->edge_id; P.op_out = o; P.mach_out = mc;
        P.mfea1 = mfea1; P.mmask = mach_mask;
        int rf = fill_obs(h, P, task_fea, mach_fea, adj_w, adj_src, job_mask, candidate, mask_mode, dtype);
        if (rf) return rf;
        P.obs_inc = obs_inc_now(h, task_fea, mach_fea, adj_w, adj_src, dtype);
        rf = dtype == MTFJSP_F64 ? launch_random_fused<double>(h, P, (cudaStream_t)stream)
                                 : launch_random_fused<float>(h, P, (cudaStream_t)stream);
        if (rf > 0) obs_mark(h, task_fea, mach_fea, adj_w, adj_src, dtype);
        if (rf != 0) return rf < 0 ? rf : MTFJSP_OK;
    }
    rc = flush_reset(h, (cudaStream_t)stream);  // the separate kernels below read the state
    if (rc) return rc;
    rc = launch_prestep<true>(h, seed, env_offset, mask_mode == MTFJSP_MASK_ESA ? h->jm_esa : h->jm_fin, o, mc, mfea1,
                                  mach_mask, dtype, (cudaStream_t)stream);
    if (rc < 0) return rc;
    if (rc == 0) {
        rc = mtfjsp_policy_random(h, seed, env_offset, mask_mode, o, mc, stream);
        if (rc) return rc;
        if (mfea1) {
            rc = mtfjsp_mfea1(h, o, mfea1, mach_mask, dtype, stream);
            if (rc) return rc;
        }
    }
    return mtfjsp_step_obs(h, o, mc, reward5, scaled4, done, invalid, task_fea, mach_fea, adj_w, adj_src, job_mask,
                           candidate, mask_mode, dtype, stream);
}

}  // extern "C"

// Host-buffer step behind both entry points.  Packed form: act [B,2] i32 in, rec [B] records out; split form: op / mach
// in, info6 / job_mask / candidate out (each may be NULL).
struct HostIO {
    const int32_t *op, *mach, *act;
    double* info6;
    uint8_t* jm;
    int32_t* cand;
    unsigned char* rec;
};

static int host_step_impl(mtfjsp_env* h, const HostIO& io, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src,
                          int mask_mode, int dtype, cudaStream_t s) {
    const Layout& L = h->L;
    const bool packed = io.act != nullptr;
    const int inc = obs_inc_now(h, task_fea, mach_fea, adj_w, adj_src, dtype);
    // In place: when every buffer the call passes is pinned and mapped into the device's address space, ONE launch over
    // the whole batch reads and writes them through their device addresses, so the PCIe writes of the first warps run
    // under the rest of the kernel -- no staging buffer, no copy engine.
    bool mapped = true;
    auto dev = [&](const void* p) -> void* {
        void* d = nullptr;
        if (p && mapped && (cudaHostGetDevicePointer(&d, const_cast<void*>(p), 0) != cudaSuccess || !d)) {
            cudaGetLastError();  // pageable, or not mapped for this device
            mapped = false;
        }
        return d;
    };
    const int2* act = reinterpret_cast<const int2*>(dev(io.act));
    const int32_t* op = reinterpret_cast<const int32_t*>(dev(io.op));
    const int32_t* mach = reinterpret_cast<const int32_t*>(dev(io.mach));
    double* info6 = reinterpret_cast<double*>(dev(io.info6));
    uint8_t* jm = reinterpret_cast<uint8_t*>(dev(io.jm));
    int32_t* cand = reinterpret_cast<int32_t*>(dev(io.cand));
    unsigned char* rec = reinterpret_cast<unsigned char*>(dev(io.rec));
    if (!mapped) {  // staged: copy in, one launch into the handle's device scratch, copy out, in order on `s`
        info6 = io.info6 ? h->info6 : nullptr;
        rec = io.rec ? h->rec : nullptr;
        jm = nullptr;  // copied out of the kernel's own mask / candidate buffers
        cand = nullptr;
    }
    // the actions are read in place from 16,384 envs up; below that the explicit copy is as fast
    if (!mapped || !h->host_act_in_place) {
        if (packed) {
            CK(cudaMemcpyAsync(h->act2, io.act, (size_t)L.B * 8, cudaMemcpyHostToDevice, s), "H2D actions");
            act = h->act2;
        } else {
            CK(cudaMemcpyAsync(h->a_op, io.op, (size_t)L.B * 4, cudaMemcpyHostToDevice, s), "H2D op");
            CK(cudaMemcpyAsync(h->a_mach, io.mach, (size_t)L.B * 4, cudaMemcpyHostToDevice, s), "H2D mach");
            op = h->a_op;
            mach = h->a_mach;
        }
    }
    int rc = launch_step_obs(h, op, mach, nullptr, nullptr, h->dn, h->inv, info6, task_fea, mach_fea, adj_w, adj_src, jm,
                             cand, mask_mode, dtype, s, act, rec, inc);
    if (rc) return rc;
    if (!mapped) {
        const size_t B = (size_t)L.B;
        const uint8_t* jm_dev = mask_mode == MTFJSP_MASK_ESA ? h->jm_esa : h->jm_fin;
        if (io.rec) CK(cudaMemcpyAsync(io.rec, h->rec, B * h->rec_stride, cudaMemcpyDeviceToHost, s), "D2H records");
        if (io.info6) CK(cudaMemcpyAsync(io.info6, h->info6, B * 48, cudaMemcpyDeviceToHost, s), "D2H info6");
        if (io.jm) CK(cudaMemcpyAsync(io.jm, jm_dev, B * L.J, cudaMemcpyDeviceToHost, s), "D2H job_mask");
        if (io.cand) CK(cudaMemcpyAsync(io.cand, h->cand, B * L.J * 4, cudaMemcpyDeviceToHost, s), "D2H candidate");
    }
    obs_mark(h, task_fea, mach_fea, adj_w, adj_src, dtype);
    CK(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return MTFJSP_OK;
}

extern "C" {

int mtfjsp_step_host(mtfjsp_env* h, const int32_t* op_host, const int32_t* mach_host, double* info6_host,
                     uint8_t* job_mask_host, int32_t* candidate_host, void* task_fea, void* mach_fea, float* adj_w,
                     int16_t* adj_src, int mask_mode, int dtype, void* stream) {
    if (!h || !op_host || !mach_host) return fail(MTFJSP_E_ARG, "mtfjsp_step_host: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_step_host before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    HostIO io = {op_host, mach_host, nullptr, info6_host, job_mask_host, candidate_host, nullptr};
    return host_step_impl(h, io, task_fea, mach_fea, adj_w, adj_src, mask_mode, dtype, (cudaStream_t)stream);
}

int mtfjsp_step_host_packed(mtfjsp_env* h, const int32_t* actions_host, void* records_host, void* task_fea, void* mach_fea,
                            float* adj_w, int16_t* adj_src, int mask_mode, int dtype, void* stream) {
    if (!h || !actions_host || !records_host) return fail(MTFJSP_E_ARG, "mtfjsp_step_host_packed: bad argument");
    if (!h->reset_done) return fail(MTFJSP_E_STATE, "mtfjsp_step_host_packed before mtfjsp_reset");
    int rc = enter(h, (cudaStream_t)stream);
    if (rc) return rc;
    HostIO io = {nullptr, nullptr, actions_host, nullptr, nullptr, nullptr, (unsigned char*)records_host};
    return host_step_impl(h, io, task_fea, mach_fea, adj_w, adj_src, mask_mode, dtype, (cudaStream_t)stream);
}

int mtfjsp_host_record_bytes(const mtfjsp_env* h) { return h ? h->rec_stride : 0; }

int mtfjsp_launch_overlap_error(const mtfjsp_env* h) { return h ? (int)*(volatile unsigned*)h->ovl_err : 0; }

int64_t mtfjsp_launch_count(const mtfjsp_env* h) { return h ? h->launches : 0; }

int64_t mtfjsp_bytes_per_gather(const mtfjsp_env* h) { return h ? (int64_t)(2 * gather_env_bytes(h->L) + 4) : 0; }

int64_t mtfjsp_bytes_per_peek(const mtfjsp_env* h, int K) { return h && K > 0 ? (int64_t)peek_env_bytes(h->L, K) : 0; }

int64_t mtfjsp_bytes_per_step(const mtfjsp_env* h, int dtype) {
    if (!h) return 0;
    // SURVEY.md 8(d): B_step = 8 (action) + 2*B_state + B_out_ell
    const int64_t N = h->L.N, M = h->L.M, J = h->L.J;
    int64_t b_state = 18 * N + 42 * M + 8 * J + (N + 7) / 8 + 160;
    int64_t fe = dtype == MTFJSP_F64 ? 8 : 4;
    int64_t b_out = 12 * fe * N + 18 * N + 8 * fe * M + 5 * J + 41;
    return 8 + 2 * b_state + b_out;
}

// SURVEY.md 8(d) accounting of the one-launch random-rollout step: the fused step + the pre-step's traffic --
// reads job mask J, candidates 4J, t / p rows 16M, edge ids M; writes the action 8 (instead of reading it), the
// candidate-machine features 6*fe*M and the machine mask M.
int64_t mtfjsp_bytes_per_random_step(const mtfjsp_env* h, int dtype) {
    if (!h) return 0;
    const int64_t M = h->L.M, J = h->L.J;
    const int64_t fe = dtype == MTFJSP_F64 ? 8 : 4;
    return mtfjsp_bytes_per_step(h, dtype) + 5 * J + 17 * M + 6 * fe * M + M;
}

int mtfjsp_random_step_is_fused(const mtfjsp_env* h) {
    if (!h || h->force_generic || !h->fuse_policy) return 0;
    return has_spec(h->L.J, h->L.M) ? 1 : 0;
}

}  // extern "C"
