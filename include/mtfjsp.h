/*
 * mtfjsp.h -- C ABI of the B200-native batched MT-FJSP disjunctive-graph environment.
 *
 * This is the drop-in boundary for the reference's batched environment hot path.  The reference
 * has no FFI (it is single-process Python); each entry point below names the Python interface it
 * replaces, so a maintainer can bind it with ctypes (see INTEGRATION.md).  "SS" abbreviates
 * graph-jsp-env/src/graph_jsp_env/disjunctive_graph_jsp_env_singlestep.py.
 *
 * Conventions
 *   - one handle per (GPU, env slice); a handle owns B environments of one size (J jobs x M ops per
 *     job = N operations, M machines, E edge groups);
 *   - every pointer is a DEVICE pointer unless the function name ends in _host; buffers are
 *     caller-owned; the library allocates only in mtfjsp_create;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and never synchronises
 *     the host, except the *_host entry points, which return after their device->host copy is done;
 *   - return value: 0 ok, negative = error (MTFJSP_E_*); nothing throws; every call that returns an
 *     error leaves its reason in mtfjsp_last_error (one message per thread);
 *   - an invalid (operation, machine) pair does not fail the batch: the env's `invalid` flag is set
 *     and its state is left untouched (the reference silently corrupts its state, SS:1495-1528);
 *   - not thread-safe per handle; handles are independent.
 *   - operation index i = job * M + position, 0-based; machines 0-based.
 *
 * Observation element type: MTFJSP_F64 reproduces the reference's float64 numpy outputs bit for bit;
 * MTFJSP_F32 is the same value rounded once to float (what the reference's networks see after their
 * `.float()` cast, model/actor_critic.py:134-158).
 */
#ifndef MTFJSP_H
#define MTFJSP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mtfjsp_env mtfjsp_env;

enum { MTFJSP_F32 = 0, MTFJSP_F64 = 1 };
enum { MTFJSP_MASK_FINISHED = 0, MTFJSP_MASK_ESA = 1 };
enum {
    MTFJSP_OK = 0,
    MTFJSP_E_ARG = -1,    /* bad argument (null handle, size out of range, ...) */
    MTFJSP_E_CUDA = -2,   /* a CUDA runtime call failed; see mtfjsp_last_error */
    MTFJSP_E_STATE = -3   /* call order violated (e.g. step before load/reset) */
};

/* Limits of this build: 2 <= M <= 64 machines, 1 <= J, N = J*M <= 4096 operations, and one environment's state must
 * fit the shared memory of one block (227 KB).  That state takes about 62*N + 8*M*M bytes, so mtfjsp_create returns
 * MTFJSP_E_ARG well below N = 4096 (no instance of 4096 operations fits).  The largest J it accepts:
 *   M = 2: J <= 1678,  M = 3: J <= 1152,  M = 7: J <= 510,  M = 32: J <= 109,  M = 33: J <= 106,  M = 64: J <= 48. */

/* replaces: Parallel_env.__init__ (trainer/parallel_env.py:19-36) + the env constructor arguments
 * perform_left_shift_if_possible / reward_function='wrk' (trainer/parallel_env.py:110-118). */
int mtfjsp_create(mtfjsp_env** h, int B, int J, int M, int E, int left_shift, int device);
int mtfjsp_destroy(mtfjsp_env* h);

/* replaces: configs weight_mk / weight_ec / weight_tt (SS:1119-1121), reward_scaling.scaling_divisor
 * (SS:1164) and GAMMA of RewardScaling (trainer/parallel_env.py:82).  Defaults 0.4/0.4/0.2, 1, 0.99. */
int mtfjsp_set_params(mtfjsp_env* h, double w_mk, double w_ec, double w_tt, double scaling_divisor, double gamma);

/* replaces: Parallel_env.get_batch (trainer/parallel_env.py:39-63).
 * t, p: [B,N,M] f64 (negative = infeasible machine); tt: [B,M,M] f64; edge: [B,E,W] int32 machine ids of
 * each edge group padded with -1. */
int mtfjsp_load(mtfjsp_env* h, const double* t, const double* p, const double* tt, const int32_t* edge, int W,
                void* stream);

/* replaces: Parallel_env.init_RewardScaling_sameBATCH (trainer/parallel_env.py:70-83) and
 * RewardScaling.reset called per episode by Run.py:283-284. */
int mtfjsp_scaler_init(mtfjsp_env* h, void* stream);
int mtfjsp_scaler_reset(mtfjsp_env* h, void* stream);

/* replaces: Parallel_env.init_DGFJSPEnv_state0 / env.reset (trainer/parallel_env.py:87-142, SS:1183-1245).
 * weights: [B,3] f64 per-env reward weights (mk, ec, tt) -- the reference draws them from python's
 * global `random` (SS:1253-1270); here they are data.
 * Every reset after the first one since a load may be deferred: it is recorded, with mtfjsp_scaler_reset if that
 * follows, and performed by the next call on the handle, on that call's stream -- inside the step launch where it can,
 * otherwise before that call's own work.  So `weights` must stay valid and unchanged until the next call on the
 * handle returns.  MTFJSP_FUSED_RESET=0 in the environment at mtfjsp_create performs every reset at the call. */
int mtfjsp_reset(mtfjsp_env* h, const double* weights, void* stream);

/* replaces: the transition + reward + reward-scaling half of Parallel_env.DGFJSPEnv_paral_step
 * (trainer/parallel_env.py:217-261; SS:716-974).
 * op, mach: [B] int32.  Outputs (any may be NULL): reward5 [B,5] f64 = (r, r_mk, r_idle, r_pt, r_tt);
 * scaled4 [B,4] f64 = running-std scaled (mk, idle, pt, tt); done [B] u8; invalid [B] u8. */
int mtfjsp_step(mtfjsp_env* h, const int32_t* op, const int32_t* mach, double* reward5, double* scaled4,
                uint8_t* done, uint8_t* invalid, void* stream);

/* replaces: the observation half of env.step / env.reset (SS:2001-2515) and the job mask + candidate
 * bookkeeping (algorithm/ppo_algorithm.py:202-317, :1126-1165).
 * dtype selects the element type of task_fea / mach_fea (MTFJSP_F32 | MTFJSP_F64).  Any output may be NULL.
 *   task_fea [B,N,12]   (est_st, est_ft, est_pt, scheduled, in_degree, machine+1, t, p, job+1, w0, w1, w2)
 *   mach_fea [B,M,8]    (ft of last op, sum pt/N, sum transport, sum idle, count, w0, w1, w2)
 *   adj_w    [B,N,2] f32  adjacency in compact ELL form: row = destination op v; [0] = weight of the arc from
 *                         its job predecessor v-1, [1] = weight of the arc from its machine predecessor
 *                         (0 = no such arc; a machine arc that coincides with the job arc is reported in [0]);
 *                         the diagonal entry is always 1 and not stored
 *   adj_src  [B,N] i16    source op of the machine-predecessor arc, -1 if none
 *   job_mask [B,J] u8     1 = job not selectable;  candidate [B,J] i32 = next op of each job
 *   mask_mode: MTFJSP_MASK_ESA (the reference's rule) or MTFJSP_MASK_FINISHED. */
int mtfjsp_obs(mtfjsp_env* h, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src, uint8_t* job_mask,
               int32_t* candidate, int mask_mode, int dtype, void* stream);

/* mtfjsp_step followed by mtfjsp_obs in one kernel launch: the state is read once. */
int mtfjsp_step_obs(mtfjsp_env* h, const int32_t* op, const int32_t* mach, double* reward5, double* scaled4,
                    uint8_t* done, uint8_t* invalid, void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src,
                    uint8_t* job_mask, int32_t* candidate, int mask_mode, int dtype, void* stream);

/* replaces: Parallel_env.cal_cur_task_machine_feature (trainer/parallel_env.py:152-214) and the machine
 * mask gather of Run.py:262-266, 335-337.  op [B] int32; mfea1 [B,M,6] (dtype); mach_mask [B,M] u8, 1 = infeasible. */
int mtfjsp_mfea1(mtfjsp_env* h, const int32_t* op, void* mfea1, uint8_t* mach_mask, int dtype, void* stream);

/* compatibility view: dense adjacency adj[b,dst,src], diagonal 1 (SS:2019-2073), element type dtype. */
int mtfjsp_dense_adj(mtfjsp_env* h, void* adj, int dtype, void* stream);

/* replaces: Instance_Dataset's sample generation (instance/generate_allsize_mofjsp_dataset.py:161-273) for synthetic
 * batches -- the same distributions drawn on the device from a counter-based generator keyed by (seed, env_offset + b),
 * so a rank generates its own slice without touching the host.  t, p [B,N,M] f64; tt [B,M,M] f64; edge [B,E,W] i32
 * (machine ids of each edge group, padded with -1; W >= largest group).  Needs J >= M.  No handle: the arrays are the
 * caller's and go to mtfjsp_load. */
int mtfjsp_generate_instances(int B, int J, int M, int E, uint64_t seed, uint64_t env_offset, double* t, double* p, double* tt,
                              int32_t* edge, int W, void* stream);

/* compatibility view of the single-env class: raw arc weights between real ops, adj[b,u,v] = trunc(weight of u -> v),
 * int32 [B,N,N] -- nx.to_numpy_array(G)[1:-1,1:-1].astype(int) of SS:2019, the matrix the reference's gym `state`
 * vector (first element of the reset 9-tuple / step 14-tuple, SS:2075-2130, 2515) is built from. */
int mtfjsp_raw_adj(mtfjsp_env* h, int32_t* adj, void* stream);

/* replaces: reading env.makespan_previous_step, total_e1_previous_step/N, trans_t_previous_step,
 * idle_t_previous_step (Run.py:632-633, trainer/validate.py:273-277).  cost4 [B,4] f64 (mk, pt/N, tt, idle);
 * total_e1 [B] f64 = the undivided total_e1_previous_step.  Either may be NULL. */
int mtfjsp_costs(mtfjsp_env* h, double* cost4, double* total_e1, void* stream);

/* parity checks / rendering: machine assignment (-1 unassigned) [B,N] i32, start / finish [B,N] f64 (0 while
 * unscheduled), machine routes [B,M,N] i32 padded with -1 (replaces env.machine_routes, env.G.nodes[...]). */
int mtfjsp_export_state(mtfjsp_env* h, int32_t* mach, double* st, double* ft, int32_t* routes, void* stream);
int mtfjsp_export_scaler(mtfjsp_env* h, double* R, double* mean, double* S, int64_t* n, void* stream);

/* Copies environments between handles: afterwards env b of `dst` is in exactly the state env idx[b] of `src` was in,
 * and every later call on dst env b returns the same bits as on a fresh env that replayed idx[b]'s whole history --
 * steps, observations, masks, candidates, rewards, scaled rewards, costs, export_state / export_scaler, and later
 * resets back to that instance.  Per env it copies the state records, the static tables (t, p, transport table,
 * minimum durations, edge groups), the reset snapshot, both job-mask forms, the candidates and the done / invalid
 * flags; dst takes src's loaded / reset status.  idx: [dst.B] int32 on the device; duplicates and permutations are
 * allowed and dst.B may differ from src.B.  The reward scaler's state travels with the env.
 * Both handles first perform a recorded reset (mtfjsp_reset): one recorded on src is in the copied state, and one
 * recorded on dst is performed before the copy overwrites it (a later step of dst would otherwise perform it on the
 * copied state).  The next step of either handle waits for the copy in full, and dst's next observation-writing step
 * rewrites every row.
 * MTFJSP_E_ARG, nothing written: src == dst, a NULL argument, different devices, (J, M, E, left_shift) differ, or the
 * mtfjsp_set_params values differ.  MTFJSP_E_STATE, nothing written: src was never loaded.  An idx[b] outside [0, src.B)
 * cannot be checked on the host without a synchronisation: for such a b the kernel writes only dst's invalid flag of
 * env b (1) and leaves the rest of that env as it was (the convention of an invalid action); debug builds
 * (MTFJSP_DEBUG_BOUNDS) assert.  src and dst must be used on the same stream, or ordered by the caller. */
int mtfjsp_gather(mtfjsp_env* dst, const mtfjsp_env* src, const int32_t* idx, void* stream);

/* One-step lookahead: for K (op, machine) pairs per env, what mtfjsp_step would return for that action from the current
 * state, without changing the state.  op, mach: [B,K] int32 on the device.  reward5 [B,K,5] f64 receives, bit for bit,
 * what the step would write for env b and action (op[b,k], mach[b,k]): r (the mtfjsp_set_params-weighted sum over the
 * divisor), then r_mk, r_idle, r_pt, r_tt.  invalid [B,K] u8 receives the step's invalid flag for the pair (the op is
 * not the next op of its job, the machine is out of range or infeasible (t < 0), or the env is done); an invalid pair
 * gets zeros in reward5, as the step writes.  Either output may be NULL.  No scaled rewards: the reward scaler does not
 * advance.
 * Read-only: nothing of the handle is written -- state records, reward-scaler state, reset snapshot, both job-mask forms,
 * candidates, done / invalid flags -- and a fused step after a peek still rewrites only the observation rows it changes.
 * A non-step call: a recorded reset (mtfjsp_reset) is performed first, so a peek right after mtfjsp_reset sees the reset
 * state, and the next step waits for the peek in full.
 * Replaces the reference's lookahead by replay (tester/pdrs.py:425-433, 495-510: reset, replay the chosen prefix, step
 * one candidate, read r_idle -- once per candidate per decision).
 * MTFJSP_E_ARG, nothing written: a NULL handle, op or mach, or K < 1.  MTFJSP_E_STATE, nothing written: before the first
 * mtfjsp_reset.  op / mach entries are data: out-of-range values make that pair invalid. */
int mtfjsp_peek(mtfjsp_env* h, const int32_t* op, const int32_t* mach, int K, double* reward5, uint8_t* invalid,
                void* stream);

/* Whole-episode replay: for R candidate action sequences, what T steps from an episode start would leave, without
 * changing the handle.  src [R] int32: candidate r starts from the episode start (the reset snapshot, which travels with
 * mtfjsp_gather) of env src[r]; actions [R,T,2] int32 (op, machine), contiguous per candidate; 1 <= T <= N.  All on the
 * device.  Outputs, any of which may be NULL: cost4 [R,4] f64 receives what mtfjsp_costs would return after the T
 * actions; return5 [R,5] f64 the step-order FP64 sum, from 0.0, of the reward5 every step would write; first_invalid [R]
 * int32 -1 if every action was valid, else the index of the first invalid one (an invalid action is a no-op, as in
 * mtfjsp_step, and the replay goes on).  The bits equal those of a fresh copy of env src[r] taken at its episode start
 * and stepped T times by mtfjsp_step, then read by mtfjsp_costs.  Rewards use the mtfjsp_set_params values; the reward
 * scaler takes no part.  A src[r] outside [0, B) is data: that candidate gets -2 in first_invalid and zero rows in
 * cost4 / return5, and the others are unaffected.
 * Read-only: nothing of the handle is written.  A non-step call: a recorded reset (mtfjsp_reset) is performed first, and
 * the next step waits for the replay in full.
 * MTFJSP_E_ARG, nothing written: a NULL handle, src or actions, R < 1, T < 1 or T > N.  MTFJSP_E_STATE, nothing written:
 * before the first mtfjsp_reset since mtfjsp_load. */
int mtfjsp_replay(mtfjsp_env* h, const int32_t* src, int R, const int32_t* actions, int T, double* cost4, double* return5,
                  int32_t* first_invalid, void* stream);

/* Neighbour replay: mtfjsp_replay of R single-move neighbours of Q base sequences, without writing the neighbours.
 * base [Q,N,2] int32 holds Q complete (op, machine) sequences, contiguous per row; base_src [Q] int32 the env whose
 * episode start row q is replayed from; moves [R,4] int32 (row, kind, s, arg): kind 0 (reassignment) runs entry s of
 * base row `row` on machine arg, kind 1 (insertion) removes entry s and inserts it at index arg of the remaining N - 1
 * (search.neighbour_moves / search.apply_moves).  All on the device.  Candidate r is replayed over all N steps; the
 * outputs are mtfjsp_replay's (any may be NULL) and their bits equal mtfjsp_replay with src = base_src[moves[:,0]] and
 * the neighbour sequences apply_moves would build, T = N.  A malformed move is data: a row outside [0, Q), a kind other
 * than 0 or 1, s outside [0, N), an insertion with arg outside [0, N), or base_src[row] outside [0, B) gives -2 in
 * first_invalid and zero rows in cost4 / return5, and the other moves are unaffected.  A reassignment to an infeasible
 * or out-of-range machine, and an insertion that breaks job order, are well-formed: they replay, and their first
 * invalid action is reported as mtfjsp_replay reports it.
 * Read-only and a non-step call, as mtfjsp_replay.
 * MTFJSP_E_ARG, nothing written: a NULL handle, base_src, base or moves, Q < 1 or R < 1.  MTFJSP_E_STATE, nothing
 * written: before the first mtfjsp_reset since mtfjsp_load. */
int mtfjsp_replay_moves(mtfjsp_env* h, const int32_t* base_src, int Q, const int32_t* base, const int32_t* moves, int R,
                        double* cost4, double* return5, int32_t* first_invalid, void* stream);

/* Episode completion: for R candidates, what the rest of the episode costs when T forced actions and then a base policy
 * finish the schedule, without changing the handle.  Candidate r starts from the CURRENT state of env src[r] (src [R]
 * int32; duplicates and permutations allowed), runs actions [R,T,2] int32 (op, machine), 0 <= T <= N (NULL when T = 0;
 * an invalid forced action is a no-op, as in mtfjsp_step, and the run goes on), then one base action at a time until
 * every op is scheduled.  The selectable jobs are those the mask_mode job mask leaves open after the same steps (the
 * mask mtfjsp_policy_random reads).
 *   MTFJSP_BASE_RANDOM: mtfjsp_policy_random's draws with env_offset 0 and env index r: the k-th selectable job by
 *     draw (seed, r, ops scheduled, stream 0), the k-th feasible machine by stream 1.  key / key_mach are not read.
 *   MTFJSP_BASE_PRIORITY: the selectable job whose candidate op c has the smallest key[src[r], c] ([B,N] f64; -0.0 equals
 *     +0.0, NaN ranks above +inf), ties to the lowest job index, on machine key_mach[src[r], c] ([B,N] int32).
 * A base action that is invalid (e.g. an infeasible key_mach entry) is data: the completion stops there.
 * Outputs, any of which may be NULL: cost4 [R,4] f64 what mtfjsp_costs would return after the run; return5 [R,5] f64 the
 * step-order FP64 sum, from 0.0, of the reward5 of every step, forced and base; first_invalid [R] int32 -1 if every action
 * was valid, else the index of the first invalid one (T + i for the i-th base action); base_actions [R,N,2] int32 the
 * base policy's actions in order, padded with -1.  The bits equal those of: mtfjsp_gather into an R-env handle with
 * idx = src, T mtfjsp_step calls with the forced actions, then mtfjsp_policy_random(seed, 0, mask_mode) (or the priority
 * choice) and mtfjsp_step until done, then mtfjsp_costs.  A src[r] outside [0, B) is data: -2 in first_invalid, zero
 * rows in cost4 / return5 and -1 in base_actions.
 * Read-only: nothing of the handle is written.  A non-step call: a recorded reset (mtfjsp_reset) is performed first, and
 * the next step waits for the completion in full.
 * MTFJSP_E_ARG, nothing written: a NULL handle or src, R < 1, T outside [0, N], T > 0 with NULL actions, a bad base or
 * mask_mode, or MTFJSP_BASE_PRIORITY with a NULL key or key_mach.  MTFJSP_E_STATE, nothing written: before the first
 * mtfjsp_reset since mtfjsp_load. */
enum { MTFJSP_BASE_RANDOM = 0, MTFJSP_BASE_PRIORITY = 1 };
int mtfjsp_complete(mtfjsp_env* h, const int32_t* src, int R, const int32_t* actions, int T, int base, const double* key,
                    const int32_t* key_mach, uint64_t seed, int mask_mode, double* cost4, double* return5,
                    int32_t* first_invalid, int32_t* base_actions, void* stream);

/* Uniform random valid action from the env's current masks: a selectable job (under mask_mode), its candidate
 * op, and a feasible machine for it; counter-based, keyed by (seed, env_offset + env, ops scheduled so far).
 * Mirrors tester/pdrs.py Random_task / Random_m (:75-86, :139-156).  op, mach [B] int32 (-1 when done). */
int mtfjsp_policy_random(mtfjsp_env* h, uint64_t seed, uint64_t env_offset, int mask_mode, int32_t* op,
                         int32_t* mach, void* stream);

/* One whole pass of the environment side of a rollout step in one launch sequence on `stream`:
 * policy_random -> mfea1 -> step_obs.  mfea1 / mach_mask may be NULL. */
int mtfjsp_random_step(mtfjsp_env* h, uint64_t seed, uint64_t env_offset, int32_t* op, int32_t* mach, void* mfea1,
                       uint8_t* mach_mask, double* reward5, double* scaled4, uint8_t* done, uint8_t* invalid,
                       void* task_fea, void* mach_fea, float* adj_w, int16_t* adj_src, uint8_t* job_mask,
                       int32_t* candidate, int mask_mode, int dtype, void* stream);

/* Incremental observation (off by default).  When on, a fused step (mtfjsp_step_obs / mtfjsp_random_step /
 * mtfjsp_step_host*) whose four observation pointers and dtype are the ones that received the previous observation
 * rewrites only the rows the step changed -- the stepped job's rows from the stepped op on, the op that now follows it
 * on its machine, the rows of the previous step's one-step transients, one machine row -- instead of all N + M rows;
 * the buffers end up bit-identical to a full rewrite.  The library tracks the chain (a reset, a load, an mtfjsp_step
 * without observation or different pointers force the next fused step to write everything); the CALLER promises not
 * to modify those buffers between steps.  The reference rebuilds every array every step (SS:2001-2515, 69 % of its
 * step time). */
int mtfjsp_set_obs_incremental(mtfjsp_env* h, int on);

/* Host-buffer form of mtfjsp_step_obs, the call a host-side rollout loop (Run.py:411-443) makes:
 * actions come from (pinned) host memory, the step info the host consumes comes back --
 * info6 [B,6] f64 = (r, done, mk_s, idle_s, pt_s, tt_s) exactly as trainer/parallel_env.py:260,
 * job_mask [B,J] u8 and candidate [B,J] i32 -- while the observation tensors stay on the device
 * (device pointers, may be NULL) for the encoder.  Synchronises `stream` before returning. */
int mtfjsp_step_host(mtfjsp_env* h, const int32_t* op_host, const int32_t* mach_host, double* info6_host,
                     uint8_t* job_mask_host, int32_t* candidate_host, void* task_fea, void* mach_fea, float* adj_w,
                     int16_t* adj_src, int mask_mode, int dtype, void* stream);

/* Packed form of mtfjsp_step_host, one copy each way: `actions_host` [B,2] i32 is the reference's joint-action list
 * [(task_idx, machine_idx), ...] (trainer/parallel_env.py:217-232) as an array; `records_host` receives B records of
 * mtfjsp_host_record_bytes(h) bytes each (8-byte aligned):
 *     f64 r, f64 scaled[4] = (mk_s, idle_s, pt_s, tt_s)     trainer/parallel_env.py:260 (oenv_info columns 0, 2..5)
 *     u8  done                                              (oenv_info column 1)
 *     u8  mask_bits[(J+7)/8]   bit (j & 7) of byte (j >> 3) set = job j not selectable   algorithm/ppo_algorithm.py:202-317
 *     u8  next_op[J]           candidate op of job j = j * M + next_op[j]; then zero padding to a multiple of 8
 * (48 bytes at J = 6: the step's D2H traffic is what bounds the call, see DESIGN.md section 5).
 * With pinned buffers (cudaHostAlloc / cudaHostRegister'd, hence mapped into the device's address space) the step is
 * ONE launch whose warps write their finished records straight into `records_host` over PCIe while the rest of the
 * batch is still being stepped -- no staging buffer, no copy engine; from 16,384 envs up the actions are read from
 * `actions_host` in place as well (below that they are copied in first).  mtfjsp_step_host writes its step info, job
 * mask and candidates into mapped buffers the same way.  If any buffer is pageable (not mapped), the call copies in,
 * steps into device scratch and copies out, in order on `stream`.  Synchronises `stream` before returning: the host
 * buffers are complete when the call returns. */
int mtfjsp_step_host_packed(mtfjsp_env* h, const int32_t* actions_host, void* records_host, void* task_fea, void* mach_fea,
                            float* adj_w, int16_t* adj_src, int mask_mode, int dtype, void* stream);
int mtfjsp_host_record_bytes(const mtfjsp_env* h);

/* ---- encoder side (SURVEY.md 8 a13) --------------------------------------------------------------------------
 * replaces: actor_critic.py:139-140 (dense adj -> sparse COO), gcn_mlp.py:125 (FP64 SpMM A*h) and :133-149 (degree
 * SpMM): out[b,v,:] = (h[b,v,:] + adj_w[b,v,0]*h[b,v-1,:] + adj_w[b,v,1]*h[b,adj_src[b,v],:]) / in_degree, FP32
 * fused multiply-adds.  h, out: [B,N,C] f32 (C % 4 == 0); adj_w / adj_src as written by mtfjsp_obs.
 *
 * Alignment (every mtfjsp_enc_* entry point below): the kernels move activations, weights and affines 16 bytes at a
 * time (float4, cp.async, TMA), so these pointers must be 16-byte aligned: h / g / x / gy / out / y / dx / mean / rstd /
 * t / dt / dparts and the BatchNorm w / b of aggregate, aggregate_bwd, bn_fwd, bn_bwd and gat_attend(_bwd); in_scale /
 * in_shift of aggregate(_grouped) and of every *_grouped layer and head; X, W, Z of the linear layers; X, Wa, W1,
 * bias_env of the heads; dY, X, workspace of wgrad; fea2, Wt, out of the GAT trunks; W0f, W1, bias_env of the ESA head.
 * adj_w, fea1 and the f64 stats / workspace / env_stats / sums buffers must be 8-byte aligned.  A misaligned pointer
 * returns MTFJSP_E_ARG before anything is launched.  Every torch allocation and every row slice of a [rows, C % 4 == 0]
 * tensor satisfies this. */
int mtfjsp_enc_aggregate(const float* h, const float* adj_w, const int16_t* adj_src, float* out, int64_t B, int N,
                         int C, const float* in_scale, const float* in_shift, int in_relu, void* stream);
/* Backward of mtfjsp_enc_aggregate for the PPO update (ppo_algorithm.py:739-775 re-runs the encoder with gradients;
 * torch autograd does the transposed FP64 SpMM there).  mtfjsp_enc_ell_invert builds the machine-successor index
 * adj_dst [B,N] i16 (-1 = none) from adj_src once per stored step; mtfjsp_enc_aggregate_bwd then computes
 * out[b,u,:] = g[b,u,:]/deg[u] + w_job[u+1]*g[b,u+1,:]/deg[u+1] + w_mach[d]*g[b,d,:]/deg[d], d = adj_dst[b,u]. */
int mtfjsp_enc_ell_invert(const int16_t* adj_src, int16_t* adj_dst, int64_t B, int N, void* stream);
int mtfjsp_enc_aggregate_bwd(const float* g, const float* adj_w, const int16_t* adj_src, const int16_t* adj_dst, float* out,
                             int64_t B, int N, int C, void* stream);
/* Grouped BatchNorm1d with batch statistics (+ optional ReLU), forward and backward, for the batched PPO re-forward:
 * x [G,R,C] f32, every one of the G row groups (= buffered steps) normalised with its own biased batch variance, as
 * the reference's per-step BatchNorm1d calls do in training mode (gcn_mlp.py:154,248; actor_critic.py:434 inside
 * ppo_algorithm.py:739-775).  C % 4 == 0.  fwd: y [G,R,C], mean / rstd [G,C] kept for the backward, workspace
 * [G,2,C] f64.  bwd: dx [G,R,C]; sums [G,2,C] f64 = per group (sum of g', sum of g'*xhat), whose sums over G are the
 * gradients of beta and gamma; g' = gy masked by y > 0 when relu. */
int mtfjsp_enc_bn_fwd(const float* x, const float* w, const float* b, float eps, int64_t G, int64_t R, int C, int relu, float* y,
                      float* mean, float* rstd, double* workspace, void* stream);
int mtfjsp_enc_bn_bwd(const float* x, const float* gy, const float* w, const float* b, const float* mean, const float* rstd,
                      int64_t G, int64_t R, int C, int relu, float* dx, double* sums, void* stream);
/* replaces: gcn_mlp.py:192 graph mean pooling; h [B,N,C] f32 -> out [B,C] f32.
 * Both take an optional per-column affine (+ReLU) applied to h on the fly: the BatchNorm of the producing layer
 * (gcn_mlp.py:154-157) folded into its consumer.  in_scale / in_shift [C] f32 or both NULL. */
int mtfjsp_enc_graph_mean(const float* h, float* out, int64_t B, int N, int C, const float* in_scale,
                          const float* in_shift, int in_relu, void* stream);
/* The machine-node trunk up to the mean over the two node sets (actor_critic.py:381-420) in one launch, hidden = 128:
 * input projections fea1 [R,6] W1p[128,6]^T and fea2 [R,8] W2p[128,8]^T, three GAT layers (projection by Wt = gat_layer.W^T
 * [128 out,128 in] on tcgen05.mma kind::tf32, attention with a_src / a_dst, ELU between layers) and the node-set mean ->
 * out [R,128]; stats (may be NULL) [256] f64 += column sums of out and of out^2 for the BatchNorm that follows
 * (actor_critic.py:434; mtfjsp_enc_bn_finalize turns them into the affine its consumers apply).  128 machines stay on one
 * SM through all three layers. */
int mtfjsp_enc_gat_trunk_tf32(const float* fea1, const float* fea2, const float* W1p, const float* W2p, const float* Wt,
                              const float* a_src, const float* a_dst, float* out, double* stats, int64_t R, void* stream);
/* One GAT layer after its projection, as the PPO update's forward runs it (hidden = 128, every pointer 16-byte aligned):
 * everything of GATLayer.forward after the projection (model/gat.py:82-159, closed form on the 2-node graph) and the
 * ELU / node-set mean around it (actor_critic.py:400-420): t [2R,128] = [t1; t2] ->
 * mode 0: [h1'; h2'], mode 1: [elu(h1'); elu(h2')], mode 2: out [R,128] = (h1' + h2') / 2. */
int mtfjsp_enc_gat_attend(const float* t, const float* a_src, const float* a_dst, float* out, int64_t R, int mode,
                          void* stream);
/* Backward of mtfjsp_enc_gat_attend for the PPO update: g = gradient of its output, dt [2R,128] = gradient of t,
 * dparts [mtfjsp_enc_gat_attend_bwd_blocks(R)][2][128] = per-block partial gradients of (a_src, a_dst) to be summed. */
int mtfjsp_enc_gat_attend_bwd(const float* t, const float* a_src, const float* a_dst, const float* g, float* dt, float* dparts,
                              int64_t R, int mode, void* stream);
int mtfjsp_enc_gat_attend_bwd_blocks(int64_t R);
/* Action selection of a rollout step (algorithm/agent_func.py:22-63): prob [B,R] = softmax over the entries with
 * mask == 0 of scores * scale (R <= 32), action [B] = a draw from it (counter-based uniform keyed by seed, *counter -- a
 * device step counter the caller advances, so that CUDA-graph replays draw fresh numbers --, env and stream_id) or the
 * first arg-max when greedy, log_a [B] = log prob[action], task [B] (may be NULL) = cand[b][action] (cand may be NULL).
 * Replaces masked_fill + softmax + torch.multinomial + gather + log + gather. */
int mtfjsp_enc_select(const float* scores, const uint8_t* mask, const int32_t* cand, float scale, int R, int64_t B, int greedy,
                      uint64_t seed, const int64_t* counter, int stream_id, float* prob, int64_t* action, float* log_a,
                      int64_t* task, void* stream);
/* A whole policy head (MLPActor, model/gcn_mlp.py:258-320, on the concatenated features of actor_critic.py:244-268 and
 * :455-470) in one launch, hidden = 128, both products on tcgen05.mma kind::tf32 with the intermediate kept on the SM:
 *   out[r] = tanh( tanh( act(X[src(r)]) Wa^T + bias_env[r / rows_per_env] ) W1^T + b1 ) . w2 + b2,   r < B * rows_per_env
 * src(r) = (r / rows_per_env) * nodes_per_env + cand[r] when cand != NULL (the candidate op of each job gathered from the
 * node embeddings), else r; act = x * in_scale + in_shift (then ReLU if in_relu) when in_scale != NULL (the producing
 * layer's BatchNorm), else identity; bias_env [bias_rows,128] with bias_rows = B or 1 = the first layer's bias plus its per-env column blocks
 * applied to the per-env inputs; b1 / b2 may be NULL. */
int mtfjsp_enc_head_tf32(const float* X, const int32_t* cand, int64_t B, int rows_per_env, int nodes_per_env,
                         const float* in_scale, const float* in_shift, int in_relu, const float* Wa, const float* bias_env,
                         int64_t bias_rows, const float* W1, const float* b1, const float* w2, const float* b2, float* out,
                         void* stream);
/* replaces: one Linear (+ the BatchNorm statistics pass, + the previous BatchNorm/ReLU apply pass) of
 * gcn_mlp.py:238-249 on the tensor cores (tcgen05.mma kind::tf32, FP32 accumulate in TMEM):
 * Z[rows,128] = act(X[rows,K]*in_scale+in_shift) @ W[128,K]^T + bias; stats[0:128] += column sums of Z,
 * stats[128:256] += column sums of Z^2 (FP64; may be NULL).  4 <= K <= 128, K % 4 == 0. */
int mtfjsp_enc_linear_tf32(const float* X, int64_t rows, int K, const float* W, const float* bias, const float* in_scale,
                           const float* in_shift, int in_relu, float* Z, double* stats, void* stream);
/* Neighbourhood aggregation (mtfjsp_enc_aggregate) and the layer that follows it in ONE launch, K = 128, N <= 128:
 * Z[r] = ( y[r] + w_job[r] y[r-1] + w_mach[r] y[src(r)] ) / n(r) + bias,  y = act(X) W^T,  act as in mtfjsp_enc_linear_tf32.
 * The aggregation is linear, so it is applied to the product rows in the epilogue (tiles hold whole envs) instead of to
 * the operand rows in a pass of its own: one read and one write of [B*N,128] less per GIN layer.  stats as above.
 * Returns MTFJSP_E_STATE when this form is not available (N > 128, no TMA driver entry point): run the two calls. */
int mtfjsp_enc_aggregate_linear_tf32(const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src, const float* W,
                                     const float* bias, const float* in_scale, const float* in_shift, int in_relu, float* Z,
                                     double* stats, void* stream);
/* Weight / bias gradient of that layer for the PPO update's backward pass (ppo_algorithm.py:918-1003; torch autograd
 * runs an FP32 library GEMM there): dW[128,K] = dY^T X, db[128] = column sums of dY (may be NULL), dY [rows,128] and
 * X [rows,K] row-major f32, 4 <= K <= 128, K % 4 == 0.  tcgen05.mma kind::tf32 with the reduction over rows (both
 * operands transposed while they are staged), one partial per CTA in `workspace`
 * (mtfjsp_enc_wgrad_workspace_floats(K) floats), partials added in CTA order: run-to-run deterministic.
 * The input gradient dX = dY W is mtfjsp_enc_linear_tf32 with W^T as the weight. */
int mtfjsp_enc_wgrad_tf32(const float* dY, const float* X, int64_t rows, int K, float* dW, float* db, float* workspace,
                          void* stream);
int64_t mtfjsp_enc_wgrad_workspace_floats(int K);
/* ESA machine actor (model/actor_critic.py:1207-1404 esa_Machine_Actor), hidden = 128, in two launches with no [R,128]
 * intermediate; fea1 [B*M,6], fea2 [B*M,8] f32, M rows per env.
 * mtfjsp_enc_esa_mach_stats: the moments the two BatchNorm calls of the actor need, from the raw features:
 *   moments [114] f64 = column sums of [fea1 | fea2] (14), sum of fea1 fea1^T (6x6 row-major), sum of fea2 fea2^T (8x8);
 *   env_mean [B,16] f32 = per-env mean of [fea1 | fea2] rows, columns 14, 15 zero.
 * Per-CTA FP64 partials in `workspace` (mtfjsp_enc_esa_mach_stats_workspace_doubles() doubles) added in CTA order:
 * run-to-run deterministic.  M <= 256.  Replaces the two [R,128] projections and the BatchNorm statistics passes.
 * mtfjsp_enc_esa_mach_fold: one thread per hidden column, FP64: the BatchNorm affine of both calls (biased variance
 * w_c^T Sigma w_c clamped at 0, eps) from moments over `rows` rows, W1 [128,6] / W2 [128,8] the input projections,
 * W0 [128,512] / b0 the first m_policy layer ->  Wf [128,16] = [W0a diag(sc1) W1 | W0b diag(sc2) W2 | 0 0],
 * b0f [128] = b0 + W0a sh1 + W0b sh2,  Wp [128,16] = [diag(sc1) W1 | diag(sc2) W2 | 0 0] / 2,  bp = (sh1 + sh2) / 2,
 * so that pooled = env_mean Wp^T + bp (the mean over machines of (h1 + h2) / 2).
 * mtfjsp_enc_esa_mach_head_tf32: the machine policy head, one launch, both products on tcgen05.mma kind::tf32:
 *   out[r] = 10 ( tanh( tanh( [fea1 | fea2 | 0 0][r] W0f^T + bias_env[r / M] ) W1^T + b1 ) . w2 + b2 )
 * W0f [128,16] = the first layer's h1 / h2 column blocks with the BatchNorm scales and both projections folded in,
 * bias_env [B,128] = its bias, the BatchNorm shifts and the pooled / h_pooled_o blocks applied per env; b1 / b2 may be
 * NULL.  Replaces 2 x linear + 2 x BatchNorm + concat + linear + tanh + linear + tanh + linear of the reference. */
int mtfjsp_enc_esa_mach_stats(const float* fea1, const float* fea2, int64_t B, int M, double* moments, float* env_mean,
                              double* workspace, void* stream);
int64_t mtfjsp_enc_esa_mach_stats_workspace_doubles(void);
int mtfjsp_enc_esa_mach_fold(const double* moments, int64_t rows, const float* W1, const float* W2, const float* gamma,
                             const float* beta, float eps, const float* W0, const float* b0, float* Wf, float* Wp, float* bp,
                             float* b0f, void* stream);
int mtfjsp_enc_esa_mach_head_tf32(const float* fea1, const float* fea2, int64_t B, int M, const float* W0f, const float* bias_env,
                                  const float* W1, const float* b1, const float* w2, const float* b2, float* out, void* stream);
/* BatchNorm1d with batch statistics as a per-column affine: scale = gamma/sqrt(var+eps), shift = beta - mean*scale. */
int mtfjsp_enc_bn_finalize(const double* stats, int64_t rows, const float* gamma, const float* beta, float eps,
                           float* scale, float* shift, int C, void* stream);

/* Grouped encoder layers: per-instance BatchNorm on the tcgen05 path (the reference's test-time rollouts run one instance
 * at a time with its modules in train mode, so every BatchNorm of model/gcn_mlp.py:154-157, 238-249 normalises with the
 * statistics of that one instance's rows; trainer/validate.py:60-297, algorithm/agent_func.py:22-63).  B envs of N =
 * rows_per_env rows each; a group is envs_per_group (epg) consecutive envs, G = B / epg groups (B % epg == 0), and every
 * affine in_scale / in_shift is [G,C] (C = 128), group of env b = b / epg.
 *   linear_tf32_grouped / aggregate_linear_tf32_grouped: the layers above with env-aligned tiles -- (128 / N) * N rows of
 *     whole envs for N <= 128, P = ceil(N / 128) tiles of 128 rows per env otherwise -- and, instead of the batch-wide
 *     stats, env_stats [B,P,2,128] f64: per env and tile piece the column sums of Z and of Z^2, written (no atomics, no
 *     zeroing needed), each summed over the env's rows in row order after the tile is stored.  An env's statistics and
 *     everything computed from them are therefore the same bits whatever its position in the batch.  K = 128 (TMA
 *     operand, in_scale optional) or 4 <= K <= 16, K % 4 == 0 (no input affine: the first layer); other K -> MTFJSP_E_ARG.
 *     MTFJSP_E_STATE: no TMA driver entry point, or (aggregate form) N > 128: run mtfjsp_enc_aggregate_grouped +
 *     mtfjsp_enc_linear_tf32_grouped instead.
 *   aggregate_grouped / graph_mean_grouped / head_tf32_grouped: mtfjsp_enc_aggregate / _graph_mean / _head_tf32 with the
 *     [G,C] affine (required here).
 *   bn_finalize_grouped: env_stats [B,P,2,C] -> scale, shift [G,C]; the pieces of an env, then the envs of a group are
 *     added in index order in FP64; biased variance over epg * N rows, eps and clamping as mtfjsp_enc_bn_finalize.
 * Limits: B * N <= 2^31 - 256 rows.  Bad arguments -> MTFJSP_E_ARG. */
int mtfjsp_enc_linear_tf32_grouped(const float* X, int64_t B, int rows_per_env, int K, const float* W, const float* bias,
                                   const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, float* Z,
                                   double* env_stats, void* stream);
int mtfjsp_enc_aggregate_linear_tf32_grouped(const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src,
                                             const float* W, const float* bias, const float* in_scale, const float* in_shift,
                                             int in_relu, int envs_per_group, float* Z, double* env_stats, void* stream);
int mtfjsp_enc_aggregate_grouped(const float* h, const float* adj_w, const int16_t* adj_src, float* out, int64_t B, int N, int C,
                                 const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, void* stream);
int mtfjsp_enc_graph_mean_grouped(const float* h, float* out, int64_t B, int N, int C, const float* in_scale, const float* in_shift,
                                  int in_relu, int envs_per_group, void* stream);
int mtfjsp_enc_head_tf32_grouped(const float* X, const int32_t* cand, int64_t B, int rows_per_env, int nodes_per_env,
                                 const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, const float* Wa,
                                 const float* bias_env, int64_t bias_rows, const float* W1, const float* b1, const float* w2,
                                 const float* b2, float* out, void* stream);
int mtfjsp_enc_bn_finalize_grouped(const double* env_stats, int64_t B, int rows_per_env, int envs_per_group, const float* gamma,
                                   const float* beta, float eps, float* scale, float* shift, int C, void* stream);
/* mtfjsp_enc_gat_trunk_tf32 over B envs of M machines (M <= 128) with per-env statistics: tiles of (128 / M) * M machines
 * of whole envs, out [B*M,128] as there, and instead of `stats` env_stats [B,1,2,128] f64 = per env the column sums of
 * out and of out^2 (written, no atomics; each env's rows added in row order in FP64, so the same bits at any batch
 * position).  mtfjsp_enc_bn_finalize_grouped(env_stats, B, M, ...) turns them into the [G,128] affines that
 * graph_mean_grouped and head_tf32_grouped apply: the machine trunk with per-group BatchNorm and no normalisation pass. */
int mtfjsp_enc_gat_trunk_tf32_grouped(const float* fea1, const float* fea2, const float* W1p, const float* W2p, const float* Wt,
                                      const float* a_src, const float* a_dst, float* out, double* env_stats, int64_t B, int M,
                                      void* stream);

/* replaces: the per-reward GAE of algorithm/ppo_algorithm.py:438-536 (python loop over buffered steps per stream).
 * r, v, v_next, adv: [T,B,4] f32 (streams mk, pt, tt, idle); done [T,B] f32; stats[8] f64 accumulates per-stream
 * sum and sum of squares of the advantages (allreduce it across ranks, then normalise). */
int mtfjsp_gae4(const float* r, const float* v, const float* v_next, const float* done, float* adv, double* stats, int T,
                int64_t B, float gamma, float lam, void* stream);
/* adv <- (adv - mean) / (std + 1e-5) per stream over `count` values (unbiased std), ppo_algorithm.py:485, 532. */
int mtfjsp_adv_normalize(float* adv, const double* stats, double count, int T, int64_t B, void* stream);

/* Pareto fronts over the three targets (pareto.py).  Handle-free, asynchronous on `stream`, no env state.
 * obj3 [P,3] f64 row-major points; seg [S+1] int64 CSR offsets (seg[0] = 0, non-decreasing): segment s is the point
 * range [seg[s], seg[s+1]), one instance's set.  All on the device.
 *
 * mtfjsp_pareto_filter: keep[p] = 1 iff point p of segment s is finite, no finite q of segment s dominates it (q <= p in
 * every component and q < p in one), and no finite q < p of segment s equals it in all three components (of duplicates
 * the first is kept); else 0.  Non-finite points get 0 and dominate nothing.  Pure comparisons: exact bits.  max_len
 * only sizes the grid (the kernel strides over longer segments); empty segments are allowed.  keep is written for the
 * points of every segment and nowhere else.
 * MTFJSP_E_ARG, nothing written: a NULL pointer, S < 0 or max_len < 0. */
int mtfjsp_pareto_filter(const double* obj3, const int64_t* seg, int S, int64_t max_len, uint8_t* keep, void* stream);
/* mtfjsp_hypervolume3: hv[s] = the exact hypervolume of segment s's points normalised by ref3[s] ([S,3] f64):
 * u_d = v_d / ref_d; only finite points with every u_d < 1 take part (they need not be non-dominated).  Participants
 * are ordered by u_z ascending (ties: index); slice i's area A_i is the 2-D area of the participants of z-rank <= i,
 * visited by u_x ascending (ties: u_y, then index), carrying m = min(m, u_y) from m = 1.0 and adding
 * (x_next - x_k) * (1.0 - m_k) to a sum from 0.0, x_next = 1.0 after the last.  hv = sum over i in slice order, from 0.0,
 * of A_i * (z_{i+1} - z_i), z_n = 1.0; an empty set gives 0.0.  One block per segment.  NaN for a segment of more than
 * 4096 points or a ref3 row not finite and > 0 in every component.
 * MTFJSP_E_ARG, nothing written: a NULL pointer or S < 0. */
int mtfjsp_hypervolume3(const double* obj3, const int64_t* seg, int S, const double* ref3, double* hv, void* stream);
/* mtfjsp_pareto_rank: rank[p] = the non-dominated-sorting front of point p within its segment, 0 for the first.  q
 * beats p when both are finite, q <= p in every component, and q != p or q < p (the filter's relation, a strict partial
 * order: of equal points the later falls to a later front).  rank is 0 when nothing beats p, else 1 + the largest rank
 * of the points that beat it, so rank == 0 is the filter's keep bit for bit.  INT32_MAX for a non-finite point; -2 for
 * every point of a segment of more than 4096 points.  Pure comparisons: exact.  max_len only sizes the launch (segments
 * up to max_len points are ranked in shared memory, longer ones from global memory).  One block per segment.
 * MTFJSP_E_ARG, nothing written: a NULL pointer, S < 0 or max_len < 0. */
int mtfjsp_pareto_rank(const double* obj3, const int64_t* seg, int S, int64_t max_len, int32_t* rank, void* stream);

/* Variation of (op, machine) sequences for evolutionary search (evolve.py).  Handle-free, asynchronous on `stream`.
 * t [S,N,M] f64 processing times of the S instances (t < 0: machine infeasible for the op), N = J*M; parents [P,N,2] and
 * children [C,N,2] int32 (op, machine) sequences, one contiguous run per sequence; pair [C,2] int32 the parent indices
 * of each child, inst [C] int32 its instance.  A child works on the job-sequence view (position s holds job op_s / M,
 * each op's machine apart) and is decoded with op = j*M + the number of earlier occurrences of j: every child of valid
 * parents is a complete valid sequence.  Draw k of child c is u = splitmix64(seed ^ splitmix64(c * 0x100000001B3 +
 * k * 0x9E3779B97F4A7C15)) >> 11, times 2^-53; an integer draw below n is min(floor(u * n), n - 1).
 *   pair[c,0] >= 0: POX -- job j is kept when draw j < 0.5 (j < J); positions of kept jobs take parent 1's entries, the
 *     others parent 2's non-kept jobs in parent 2's order; op o's machine is parent 1's when draw J + o < 0.5, else
 *     parent 2's.  Then with draw J+N < p_swap, positions draws J+N+1 and J+N+2 (below N) of the job sequence swap;
 *     op o with draw J+N+3+2o < p_mach takes the (draw J+N+4+2o below F)-th of its F feasible machines in machine order.
 *   pair[c,0] == -1: a random child -- draws [1, N) shuffle the job sequence 0..0 1..1 ... (each job M times) by
 *     Fisher-Yates (for i = N-1 down to 1, swap i with draw i below i+1), op o takes the (draw N+o below F)-th feasible
 *     machine; no mutation.
 * A child whose pair[c,0] is outside [-1, P), whose pair[c,1] is outside [0, P) when pair[c,0] >= 0, whose inst[c] is
 * outside [0, S), or one of whose parents holds an op outside [0, N) or a machine outside [0, M), is all -1; the other
 * children are unaffected.  Parents that are in range but not valid sequences give unspecified children.
 * MTFJSP_E_ARG, nothing written: a NULL pointer, S, P or C < 0, or (J, M) outside mtfjsp_create's range (J >= 1,
 * 2 <= M <= 64, N <= 4096). */
int mtfjsp_offspring(const double* t, int S, int J, int M, const int32_t* parents, int P, const int32_t* pair,
                     const int32_t* inst, int C, uint64_t seed, double p_swap, double p_mach, int32_t* children,
                     void* stream);

/* Monte Carlo tree search over joint (op, machine) actions (search.mcts_search).  Handle-free, asynchronous on `stream`.
 * S trees, one per instance, each a pool of P = max_nodes nodes in caller-owned device arrays: node [S,P,7] int32 holds
 * per node (parent, first_child, n_children, op, mach, visits, virtual) -- parent -1 at a tree's first root, first_child
 * -1 and n_children 0 until the node is expanded, (op, mach) the action of the edge from its parent; vmin [S,P] f64 the
 * least objective backed up through the node (+inf until then); root [S] and count [S] int32 (nodes in use, node 0 ..
 * count - 1); lohi [S,2] f64 the least and largest finite objective the tree has seen (+inf, -inf before any).  A node
 * stands for the state its path of edge actions from the root reaches; no env state is stored.
 * Children: with rule_mach == NULL, flat index j*M + m for every job j with next op k = next_op[s,j] < M (k = M: finished)
 * and every machine m with t[s, j*M+k, m] >= 0; with rule_mach [S,N] int32, flat index j on machine rule_mach[s, j*M+k]
 * when t >= 0 there.  An expanded node's valid children are one contiguous block, in flat-index order, allocated at count.
 * The job mask is MTFJSP_MASK_FINISHED's.  t [S,N,M] f64, next_op [S,J] int32 the root's state; N = J*M.
 *
 * mtfjsp_mcts_select: one warp per tree makes L selections in order l = 0 .. L-1.  A selection starts at the root; at each
 * node x, with seen = visits + virtual of x read first, virtual[x] += 1, then:
 *   unexpanded: the path ends at x when seen == 0, at depth max_depth, when x has no valid child (terminal: scored
 *     again), or when its block does not fit (count + n > P: x stays a leaf); else x is expanded and the walk steps into
 *     its first child;
 *   expanded: the lowest child with visits + virtual == 0; if none, the child of the largest score
 *     q*n/(n+v) + c*sqrt(Nx + Vx)/(1+n+v) (n, v the child's counts; Nx + Vx = seen + 1, x's counts with this path;
 *     q = 0 for vmin = +inf, else 1 when hi == lo, else (hi - vmin)/(hi - lo); FP64, evaluated in that order, no FMA),
 *     ties to the lowest child.  At depth max_depth the path ends at x.
 * paths [S*L, max_depth, 2] int32 receives row s*L + l's edge actions root-first, padded with -1; depth [S*L] its length;
 * leaf [S*L] its last node (-1 when the tree's root or count is out of range: that tree's rows are all padding and the
 * tree is not written).  A malformed block (first_child out of [0, count - n_children]) ends the path at its node.
 * mtfjsp_mcts_backup: one thread per tree takes objective [S*L] f64 (+inf for a failed completion) and, for l = 0 .. L-1
 * in order, walks from leaf[s*L+l] up the parents to the root: visits += 1, virtual -= 1, vmin = v if v < vmin; then,
 * if v is finite, lo = min(lo, v) and hi = max(hi, v).  A leaf outside [0, count) is skipped; a parent outside [0,
 * count) ends the walk.  The serial order makes the trees bit-reproducible.
 * MTFJSP_E_ARG, nothing written: a NULL pointer (rule_mach may be NULL), S < 1, L < 1, max_nodes < 1, max_depth < 0, or
 * (J, M) outside mtfjsp_create's range (J >= 1, 2 <= M <= 64, N <= 4096). */
int mtfjsp_mcts_select(const double* t, const int32_t* rule_mach, int S, int J, int M, const int32_t* next_op, int L,
                       int max_nodes, int max_depth, double c, int32_t* node, double* vmin, const int32_t* root,
                       int32_t* count, const double* lohi, int32_t* paths, int32_t* depth, int32_t* leaf, void* stream);
int mtfjsp_mcts_backup(int S, int L, int max_nodes, const int32_t* leaf, const double* objective, int32_t* node,
                       double* vmin, const int32_t* root, const int32_t* count, double* lohi, void* stream);

/* One tabu-search iteration's move for S instances, applied in place (search.tabu_search).  Handle-free, asynchronous on
 * `stream`, one warp per instance.  N = J*M.  moves [R,4] int32 (instance, kind, s, arg) are the iteration's moves in
 * search.neighbour_moves' form and order, instance s's in moves[seg[s] .. seg[s+1]) (seg [S+1] int64); obj [R] f64 their
 * objectives and f4 [R,4] f64 their final costs (moves, obj and f4 may be NULL when R = 0).  State, updated in place:
 * cur [S,N,2] int32, cur_obj [S], cur_f4 [S,4], best [S,N,2] int32, best_obj [S], best_f4 [S,4] f64; mach_until [S,N,M]
 * int32, the first iteration at which op o may again be reassigned to machine m; op_until [S,N] int32, the first
 * iteration at which op o may again be moved by insertion.  With o the op at index s of cur: a reassignment (s, m') is
 * tabu iff mach_until[o,m'] > it, an insertion iff op_until[o] > it.  A move is admissible iff it is not tabu or its
 * objective is strictly below best_obj (aspiration).  The admissible move of the least objective is taken, ties to the
 * lowest move index; a NaN objective never wins.  Taking it: cur becomes search.apply_moves(cur, move); a reassignment
 * sets mach_until[o, m_old] = it + 1 + tenure_mach, an insertion op_until[o] = it + 1 + tenure_ins; cur_obj and cur_f4
 * take the move's obj and f4; if that objective is below the previous best_obj, cur is copied to best and best_obj /
 * best_f4 take it too.  chosen [S] int32 receives the move's index in moves, -1 when the instance has no admissible move
 * (an empty segment included) and stays put, or -2 when its segment is malformed (seg[s] < 0, seg[s+1] < seg[s] or
 * seg[s+1] > R) and it stays put.  A move is never taken when its instance field is not s, its kind is not 0 or 1, s is
 * outside [0, N), its arg is outside [0, M) (reassignment) or [0, N) (insertion), or the entry of cur it names holds an
 * op outside [0, N) or, for a reassignment, a machine outside [0, M).
 * MTFJSP_E_ARG, nothing written: a NULL pointer (see above), S < 1, (J, M) outside mtfjsp_create's range (J >= 1,
 * 2 <= M <= 64, N <= 4096), R < 0 or R > INT32_MAX, it, tenure_mach or tenure_ins < 0, or it + 1 + a tenure above
 * INT32_MAX. */
int mtfjsp_tabu_move(int S, int J, int M, const int32_t* moves, int64_t R, const int64_t* seg, const double* obj,
                     const double* f4, int it, int tenure_mach, int tenure_ins, int32_t* cur, double* cur_obj,
                     double* cur_f4, int32_t* best, double* best_obj, double* best_f4, int32_t* mach_until,
                     int32_t* op_until, int32_t* chosen, void* stream);

/* Parallel tempering over finished schedules (search.anneal_search): S instances with K Markov chains each.  Handle-free,
 * asynchronous on `stream`.  N = J*M.  Chain row q = s*K + k (instance s, chain k); cur [S*K,N,2] int32 holds the rows'
 * complete (op, machine) sequences, contiguous per row.
 * Draws: chain k's draws at iteration it are u_j = evolve._draws(seed, (it << 32) | k, 3)[j], i.e.
 * x = splitmix64(seed ^ splitmix64(c * 0x100000001B3 + j * 0x9E3779B97F4A7C15)), u_j = (x >> 11) * 2^-53 with
 * c = (it << 32) | k (all mod 2^64); u0 is the proposal, u1 the Metropolis test, u2 the exchange of the pair whose lower
 * chain is k.  The instance row is not in the key, so an instance's run depends neither on the batch nor on its row.
 * below(u, n) = min(floor(u * n), n - 1) with u * n an FP64 product.
 * exp_neg(x): NaN for NaN, 1 for x <= 0, 0 for x > 746; otherwise, in FP64 with every operation correctly rounded and
 * none contracted: n = rint(x * 1.4426950408889634) (ties to even), z = -((x - n * LN2_HI) - n * LN2_LO) with
 * LN2_HI = 0x3fe62e42fee00000 (0.6931471803691238) and LN2_LO = 1.9082149292705877e-10, p = c13 and then p = p * z + c_i
 * for i = 12 .. 0 with c_i = 1/i! rounded to double, and the result scalbn(p, -n), correctly rounded (subnormals too).
 * mtfjsp_anneal_propose writes moves [S*K,4] int32 (row, kind, s, arg) in search.neighbour_moves' form with row = q.
 * Row q's neighbourhood is neighbour_moves' for its sequence and t [S,N,M] f64 (t < 0: infeasible) of instance s, in its
 * order: reassignments (s, m') for every entry s and every machine m' != m_s with t[s][o_s][m'] >= 0, in (s, m') order,
 * then insertions (s, s') for every s' in (pos(pred), pos(succ)) other than s and s - 1, in (s, s') order, where pos(pred)
 * is the index of o_s - 1 if o_s % M > 0, else -1, and pos(succ) the index of o_s + 1 if o_s % M < M - 1, else N.  With
 * R_q moves, chain q takes move number below(u0, R_q).  A row with R_q = 0, and a row whose ops are not a permutation of
 * [0, N), get (q, -1, 0, 0): a malformed move.
 * mtfjsp_anneal_step makes iteration it's decisions for every chain and applies them in place.  moves [S*K,4] int32 are
 * the proposals (row q's is moves[q]), first_invalid [S*K] int32, obj [S*K] f64 and f4 [S*K,4] f64 their replay's first
 * invalid index, objective and final costs; temp [S,K] f64 absolute temperatures (T of chain q is temp[q]).  State,
 * updated in place: cur, cur_obj [S*K], cur_f4 [S*K,4] f64; best [S,N,2] int32, best_obj [S], best_f4 [S,4] f64.
 * accepted [S*K] and swapped [S*K] int32 are written every call.  Per instance, in this order:
 *  1. Metropolis: chain q takes its proposal iff the move is well formed for row q (row == q, kind 0 or 1, s in [0, N),
 *     the op at index s of cur[q] in [0, N), and for a reassignment arg and that entry's machine in [0, M), for an
 *     insertion arg in [0, N)), first_invalid[q] == -1, obj[q] is not NaN, and delta = obj[q] - cur_obj[q] <= 0 or
 *     T > 0 and u1 < exp_neg(delta / T).  Taking it sets cur[q] = search.apply_moves(cur[q], move), cur_obj[q] = obj[q]
 *     and cur_f4[q] = f4[q].  accepted[q] = 1 if it was taken, else 0.
 *  2. Exchange, only when swap_parity is 0 or 1: for every pair a = s*K + k, b = a + 1 with k = swap_parity (mod 2) and
 *     k + 1 < K, with d = cur_obj[b] - cur_obj[a] after step 1, the pair swaps iff d <= 0, or temp[a] > 0 and
 *     u2 (of chain k) < exp_neg(d * (1 / temp[a] - 1 / temp[b])).  A swap exchanges the two rows of cur, cur_obj and
 *     cur_f4 (not the temperatures).  swapped[a] = 1 if the pair (k, k + 1) swapped; every other entry is 0.
 *  3. Best: the least cur_obj over the instance's chains that is strictly below best_obj[s], ties to the lowest k (NaN
 *     never wins), is copied with its row and cur_f4 to best[s], best_obj[s] and best_f4[s].
 * Every index and value in device memory is data and never a fault.
 * MTFJSP_E_ARG, nothing written: a NULL pointer, S < 1, K < 1, S*K > INT32_MAX, it < 0, or (J, M) outside mtfjsp_create's
 * range (J >= 1, 2 <= M <= 64, N <= 4096). */
int mtfjsp_anneal_propose(const double* t, int S, int J, int M, int K, const int32_t* cur, uint64_t seed, int it,
                          int32_t* moves, void* stream);
int mtfjsp_anneal_step(int S, int J, int M, int K, const int32_t* moves, const int32_t* first_invalid,
                       const double* obj, const double* f4, const double* temp, uint64_t seed, int it, int swap_parity,
                       int32_t* cur, double* cur_obj, double* cur_f4, int32_t* best, double* best_obj, double* best_f4,
                       int32_t* accepted, int32_t* swapped, void* stream);

/* Nonzero if a step launch of this handle waited more than 1 s for the previous one to finish the same envs
 * (MTFJSP_LAUNCH_OVERLAP) and went on; every later call on the handle then returns MTFJSP_E_CUDA.  Reads a mapped host
 * word: it reflects the launches the device has finished so far (read it after synchronising). */
int mtfjsp_launch_overlap_error(const mtfjsp_env* h);
/* Number of kernel launches issued through this handle so far (bench.py reports it). */
int64_t mtfjsp_launch_count(const mtfjsp_env* h);
/* Algorithmic bytes per env-step of the fused step+obs kernel for this handle's sizes (SURVEY.md 8d). */
int64_t mtfjsp_bytes_per_step(const mtfjsp_env* h, int dtype);
/* Same for the one-launch random-rollout step (mtfjsp_random_step on a size with a specialised kernel): the step's
 * bytes plus the policy / candidate-machine-feature traffic (job mask, candidates, t / p rows, edge ids in; action,
 * [M,6] features, machine mask out).  mtfjsp_random_step_is_fused: 1 if mtfjsp_random_step is that single launch. */
int64_t mtfjsp_bytes_per_random_step(const mtfjsp_env* h, int dtype);
/* Bytes mtfjsp_gather reads and writes per destination env (the records and tables it copies, counted once each way). */
int64_t mtfjsp_bytes_per_gather(const mtfjsp_env* h);
/* Bytes mtfjsp_peek reads and writes per env for K pairs (the record prefix it stages once, per pair the pair, its t / p
 * entries and the outputs). */
int64_t mtfjsp_bytes_per_peek(const mtfjsp_env* h, int K);
int mtfjsp_random_step_is_fused(const mtfjsp_env* h);
const char* mtfjsp_last_error(void);
const char* mtfjsp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MTFJSP_H */
