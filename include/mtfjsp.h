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
 *   - return value: 0 ok, negative = error (MTFJSP_E_*); nothing throws;
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
 * With pinned buffers (cudaHostAlloc / cudaHostRegister'd, hence mapped into the device's address space) and a
 * size-specialised kernel, the step is ONE launch whose warps write their finished records straight into
 * `records_host` over PCIe while the rest of the batch is still being stepped -- no staging buffer, no copy engine
 * (MTFJSP_HOST_ZEROCOPY: 1 = records, 2 = the actions are read from `actions_host` in place as well; default 2 from
 * 16,384 envs up, else 1; 0 = the staged form).  Staged form: the batch is cut into MTFJSP_HOST_CHUNKS (default 4) chunks
 * whose copy-in -> kernel -> copy-out chains run on three streams, replayed as one CUDA graph per step, so that the
 * copy-out of chunk c overlaps the kernel of chunk c+1; pageable buffers take the plain in-order path.  mtfjsp_step_host
 * with NULL job_mask_host / candidate_host writes its [B,6] step info the same zero-copy way.  Synchronises `stream`
 * before returning: the host buffers are complete when the call returns. */
int mtfjsp_step_host_packed(mtfjsp_env* h, const int32_t* actions_host, void* records_host, void* task_fea, void* mach_fea,
                            float* adj_w, int16_t* adj_src, int mask_mode, int dtype, void* stream);
int mtfjsp_host_record_bytes(const mtfjsp_env* h);

/* ---- encoder side (SURVEY.md 8 a13) --------------------------------------------------------------------------
 * replaces: actor_critic.py:139-140 (dense adj -> sparse COO), gcn_mlp.py:125 (FP64 SpMM A*h) and :133-149 (degree
 * SpMM): out[b,v,:] = (h[b,v,:] + adj_w[b,v,0]*h[b,v-1,:] + adj_w[b,v,1]*h[b,adj_src[b,v],:]) / in_degree, FP32
 * fused multiply-adds.  h, out: [B,N,C] f32 (C % 4 == 0); adj_w / adj_src as written by mtfjsp_obs. */
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
/* Rollout-path fusions of the machine actor and the policy heads (hidden = 128, every pointer 16-byte aligned):
 * mach_proj   replaces m_fea_1_fcl / m_fea_2_fcl (actor_critic.py:381-392) + the concatenation: fea1 [R,6], fea2 [R,8],
 *             W1 [128,6], W2 [128,8] -> out [2R,128] = [fea1 W1^T ; fea2 W2^T];
 * gat_attend  replaces everything of GATLayer.forward after the projection (model/gat.py:82-159, closed form on the
 *             2-node graph) and the ELU / node-set mean around it (actor_critic.py:400-420): t [2R,128] = [t1; t2] ->
 *             mode 0: [h1'; h2'], mode 1: [elu(h1'); elu(h2')], mode 2: out [R,128] = (h1' + h2') / 2;
 * bias_tanh   z[r] = tanh(z[r] + bias[r / rows_per_env]) in place (first layer of MLPActor, gcn_mlp.py:305-320, with the
 *             per-env part of its input applied as a bias), bias [bias_rows,128], bias_rows = rows / rows_per_env or 1;
 * tanh_dot    out[r] = tanh(z[r]) . w + b (second tanh and the Linear(128,1) of the same MLP). */
int mtfjsp_enc_mach_proj(const float* fea1, const float* fea2, const float* W1, const float* W2, float* out, int64_t R,
                         void* stream);
/* The machine-node trunk up to the mean over the two node sets (actor_critic.py:381-420) in one launch, hidden = 128:
 * input projections fea1 [R,6] W1p[128,6]^T and fea2 [R,8] W2p[128,8]^T, three GAT layers (projection by Wt = gat_layer.W^T
 * [128 out,128 in] on tcgen05.mma kind::tf32, attention with a_src / a_dst, ELU between layers) and the node-set mean ->
 * out [R,128]; stats (may be NULL) [256] f64 += column sums of out and of out^2 for the BatchNorm that follows
 * (actor_critic.py:434; mtfjsp_enc_bn_finalize turns them into the affine its consumers apply).  64 machines stay on one
 * SM through all three layers; replaces mtfjsp_enc_mach_proj + 3 x (mtfjsp_enc_linear_tf32 + mtfjsp_enc_gat_attend). */
int mtfjsp_enc_gat_trunk_tf32(const float* fea1, const float* fea2, const float* W1p, const float* W2p, const float* Wt,
                              const float* a_src, const float* a_dst, float* out, double* stats, int64_t R, void* stream);
int mtfjsp_enc_gat_attend(const float* t, const float* a_src, const float* a_dst, float* out, int64_t R, int mode,
                          void* stream);
/* Backward of mtfjsp_enc_gat_attend for the PPO update: g = gradient of its output, dt [2R,128] = gradient of t,
 * dparts [mtfjsp_enc_gat_attend_bwd_blocks(R)][2][128] = per-block partial gradients of (a_src, a_dst) to be summed. */
int mtfjsp_enc_gat_attend_bwd(const float* t, const float* a_src, const float* a_dst, const float* g, float* dt, float* dparts,
                              int64_t R, int mode, void* stream);
int mtfjsp_enc_gat_attend_bwd_blocks(int64_t R);
int mtfjsp_enc_bias_tanh(float* z, const float* bias, int64_t rows, int rows_per_env, int64_t bias_rows, void* stream);
int mtfjsp_enc_tanh_dot(const float* z, const float* w, const float* b, float* out, int64_t rows, void* stream);
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
 * applied to the per-env inputs; b1 / b2 may be NULL.  Replaces torch.gather + mtfjsp_enc_linear_tf32 +
 * mtfjsp_enc_bias_tanh + mtfjsp_enc_linear_tf32 + mtfjsp_enc_tanh_dot. */
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
int mtfjsp_random_step_is_fused(const mtfjsp_env* h);
const char* mtfjsp_last_error(void);
const char* mtfjsp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MTFJSP_H */
