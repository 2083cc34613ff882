/* ddrl_b200.h — C ABI of libddrl_b200.so (B200 / sm_100a learner hot path of DDRL).
 *
 * The reference (LucaHermes/ddrl) is pure Python on TF/RLlib and has NO FFI; this header is the
 * boundary a maintainer binds with ctypes/cffi (INTEGRATION.md shows the stub).  Each entry point
 * names the reference computation it replaces (paths relative to the reference repo root; "RLlib"
 * = ray[rllib]==1.0.1, the version README.md:47 pins).
 *
 * Conventions (all entry points):
 *   - every pointer is a DEVICE pointer to contiguous row-major memory unless it says "host";
 *     model tensors are float32, filter state float64, counts int64, indices int32, dones uint8;
 *   - shapes are explicit ints; the last argument is the cudaStream_t to launch on (as void*);
 *   - no allocation, no host synchronisation, no ownership transfer: the caller owns every buffer,
 *     including the workspaces whose sizes the *_bytes() helpers return;
 *   - return 0 on success, <0 on error (DDRL_E_*); ddrl_last_error() gives the thread-local text;
 *   - re-entrant and thread-safe per stream; ONE DEVICE PER PROCESS (the one-process-per-GPU model): kernels that need more
 *     than 48 KB of dynamic shared memory opt in once per process, on the device that is current at their first launch;
 *   - there is NO CPU fallback: without an sm_100 device every launch returns DDRL_E_CUDA.
 */
#ifndef DDRL_B200_H
#define DDRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDRL_OK 0
#define DDRL_E_BADARG (-1)
#define DDRL_E_UNSUPPORTED_SHAPE (-2)
#define DDRL_E_WORKSPACE (-3)
#define DDRL_E_CUDA (-4)

#define DDRL_HIDDEN 64      /* fcnet_hiddens = [64, 64] in every published params.json            */
#define DDRL_MAX_OBS 64     /* D <= 64  (reference: 19..44)                                        */
#define DDRL_MAX_ACT 8      /* A <= 8   (reference: 2, 4, 8)                                       */
#define DDRL_NSTAT 8        /* per-minibatch stat sums, see ddrl_ppo_train_step                    */
#define DDRL_GN_NODES 4     /* legs of the quantruped graph                                        */
#define DDRL_GN_FEATS 19    /* per-leg features, hard-coded in models/graph_net.py:16,35           */
#define DDRL_GN_ENC_IN 4    /* state[..., -4:]  models/graph_net.py:33                             */

const char* ddrl_last_error(void);
/* ABI version of this header; bumped on any signature change. */
int ddrl_abi_version(void);
/* Number of kernels this library has launched in the calling process (monotonic; for bench.py's
 * "gpu_launches" claim). */
int64_t ddrl_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * FCNet parameter layout.  One flat float32 vector per policy in the Keras/checkpoint variable
 * order of models/fcnet_glorot_uniform_init.py:48-113 with vf_share_layers=false:
 *   fc_1/kernel[D,64] fc_1/bias[64] fc_value_1/kernel[D,64] fc_value_1/bias[64]
 *   fc_2/kernel[64,64] fc_2/bias[64] fc_value_2/kernel[64,64] fc_value_2/bias[64]
 *   fc_out/kernel[64,2A] fc_out/bias[2A] value_out/kernel[64,1] value_out/bias[1]
 * = 128*D + 130*A + 8513 floats.  P policies are stored as theta[P][NP].
 * ------------------------------------------------------------------------------------------- */
int ddrl_fcnet_num_params(int D, int A);

/* Packed weight image: the FCNet kernels keep one policy's weights in shared memory in a kernel-specific
 * layout (branches concatenated, layer 2 also transposed, head matrix transposed).  An image is that layout in
 * global memory, img[P][ddrl_fcnet_image_floats(D, A)], so the per-step weight load of the SGD loop is one
 * coalesced 128-bit copy.  ddrl_fcnet_pack builds it from theta; ddrl_clip_adam keeps it in step when given.
 * Every entry point that takes (theta, img) uses img when it is not NULL and theta otherwise. */
int ddrl_fcnet_image_floats(int D, int A);
int ddrl_fcnet_pack(const float* theta, int P, int D, int A, float* img, void* stream);

/* Replaces: ray.rllib.utils.filter.MeanStdFilter.__call__ (vectorised update), instantiated at
 * simulation_envs/observation_filter.py:8-12 and by observation_filter="MeanStdFilter"
 * (train_experiment_3_architecture_curriculum_targetvel.py:71).
 * Pushes rows x[p][0..R) into the running statistics of policy p (Chan merge of fixed-order chunk
 * partials; n is exact int64) and writes norm[p] = {mean[D], 1/(std+1e-8)[D]} (float64) computed
 * from the UPDATED state, where std = sqrt(S/(n-1)) (n>1) or |M| (n<=1).
 *   x        [P][R][D] float32 (x_is_f64=0) or float64 (x_is_f64=1)
 *   n        [P] int64, M [P][D] float64, S [P][D] float64      (in/out)
 *   norm     [P][2][D] float64                                    (out)
 *   ws       workspace of ddrl_filter_ws_bytes(P, R, D) bytes
 * R == 0 only refreshes norm. */
int64_t ddrl_filter_ws_bytes(int P, int64_t R, int D);
int ddrl_filter_update(const void* x, int x_is_f64, int P, int64_t R, int D, int64_t* n, double* M,
                       double* S, double* norm, void* ws, void* stream);
/* The two halves of ddrl_filter_update, for data-parallel learners (RLlib FilterManager.synchronize:
 * worker filter buffers are merged into the driver copy): every rank runs ddrl_filter_partial on its
 * own rows, the workspaces are all-gathered and concatenated per policy in rank order to
 * parts [P][nparts][D][3] float64 = {count, mean, M2}, and ddrl_filter_merge folds them into the
 * running state in that fixed order (R_total = rows summed over all parts; n stays exact).
 * ddrl_filter_num_partials(R) = partials per policy that ddrl_filter_partial writes for R rows. */
int ddrl_filter_num_partials(int64_t R);
int ddrl_filter_partial(const void* x, int x_is_f64, int P, int64_t R, int D, void* ws, void* stream);
int ddrl_filter_merge(const void* parts, int nparts, int P, int D, int64_t R_total, int64_t* n,
                      double* M, double* S, double* norm, void* stream);

/* Replaces: the sampler's row-by-row filter calls of RLlib rollout workers (evaluation/sampler.py
 * _process_observations: one unvectorised MeanStdFilter.__call__ per observation row, i.e. RunningStat.push
 * into rs and buffer, then (x - mean) / (std + 1e-8) with the UPDATED state), W workers per policy.
 *   x        [P][R][D] float32 (x_is_f64=0) or float64 (x_is_f64=1), R = T*C rows in order t*C + c
 *            (step-major, then environment, then the agent columns of an environment)
 *   W        streams (rollout workers) per policy: stream w owns columns [w*C/W, (w+1)*C/W) and filters its
 *            rows in (t, c) order; C % W == 0
 *   n, M, S  [P] int64, [P][D], [P][D] float64: the running state every stream starts from (read only)
 *   clip     >0: clip the normalised rows to [-clip, clip]; 0: none
 *   out      [P][R][D] float32: row i normalised with its stream's state after pushing row i (float64
 *            arithmetic in the reference's operation order, one rounding to float32)
 *   parts    [P][W][D][3] float64 {count, mean, M2}: each stream's own rows (the worker's buffer), in the
 *            layout of ddrl_filter_merge.  Folding them into n/M/S in worker order (ddrl_filter_merge with
 *            R_total = R) is FilterManager.synchronize (apply_changes -> RunningStat.update).
 *   ws       workspace of ddrl_filter_stream_ws_bytes(P, T, C, W, D) bytes (<0: bad shape)
 * Fixed-order scan of chunk Welford states (no atomics): bit-identical from run to run and independent of
 * the launch geometry; the first rows of every stream match the sequential reference bit for bit, later rows
 * start from a merged state within 1e-12 relative of the sequential one.  D > DDRL_MAX_OBS returns
 * DDRL_E_UNSUPPORTED_SHAPE. */
int64_t ddrl_filter_stream_ws_bytes(int P, int T, int64_t C, int W, int D);
int ddrl_filter_stream(const void* x, int x_is_f64, int P, int T, int64_t C, int W, int D, const int64_t* n,
                       const double* M, const double* S, double clip, float* out, double* parts, void* ws,
                       void* stream);

/* Replaces: FullyConnectedNetwork_GlorotUniformInitializer.forward / value_function
 * (models/fcnet_glorot_uniform_init.py:120-125) for P grouped policies, with optional fused
 * prologue/epilogue:
 *   obs      [P][R][D] float32 raw or already-normalised observations
 *   norm     [P][2][D] float64 or NULL: if given, x = (float)((double)obs - mean) * inv)  (the
 *            MeanStdFilter output, cast to float32 as RLlib does at the policy input)
 *   clip     >0: clip normalised obs to [-clip, clip] (env-singleton filter path, clip=10); 0: none
 *   obs_out  [P][R][D] float32 or NULL: the network input actually used (stored for the SGD epochs)
 *   logits   [P][R][2A], value [P][R]                         (out; either may be NULL)
 *   eps      [P][R][A] float32 or NULL: if given, DiagGaussian sample (RLlib
 *            models/tf/tf_action_dist.py): action = mean + exp(log_std)*eps -> action [P][R][A]
 *            (unclipped, as stored in the sample batch) and logp [P][R]. */
int ddrl_fcnet_forward(const float* theta, const float* img, const float* obs, const double* norm,
                       float clip, int P, int64_t R, int D, int A, float* obs_out, float* logits,
                       float* value, const float* eps, float* action, float* logp, void* stream);

/* Replaces: distribute_observations / get_obs_indices (simulation_envs/quantruped_adaptor_multi_environment.py:124-136,
 * simulation_envs/quantruped_v3.py:282-300): per-agent index gather of the full observation, batched on the device.
 *   obs_full [S][Dfull] float32/float64 (S = env-steps), table [Ag][D] int32 (agents in agent_names order; data, not
 *   hard-coded), P policies with Ag/P agents each -> out [P][S*(Ag/P)][D] float32, row = s*(Ag/P) + j. Bit-exact. */
int ddrl_obs_gather(const void* obs_full, int is_f64, int64_t S, int Dfull, const int32_t* table, int Ag,
                    int D, int P, float* out, void* stream);

/* Replaces (batched over S env-steps): QuantrupedDecentralizedSharedGraphEnv.distribute_observations with its
 * leg_encoding_ego / quaternion_multiply (simulation_envs/quantruped_GraphDecentralizedController_environments.py:145-161,
 * 215-245): the node-feature matrix of the shared-graph policy.
 *   obs_full [S][Dfull] float32/float64 RAW observations; table [Ag][Dn] int32 (obs_indices, agent order);
 *   mean / stdv [Dfull] float64 or NULL: frozen statistics of the env-side MeanStdFilter (y = (x-mean)/(std+1e-8));
 *   clip > 0: clamp to [-clip, clip] (RLlib default 10); leg_zw [Ag][2] float64 = {sin, cos} of HALF the leg angle
 *   -> state float32: replicate == 0: [S][Ag][Dn+4];  replicate != 0: [S*Ag][Ag][Dn+4] (sample row s*Ag+j = agent j's
 *      observation tuple, all Ag rows of an env-step carry the same matrix) and node_idx [S*Ag] int32 = j (may be NULL).
 *   float64 arithmetic, rounded once to float32: bit-exact against numpy. */
int ddrl_graph_obs_build(const void* obs_full, int is_f64, int64_t S, int Dfull, const int32_t* table, int Ag,
                         int Dn, const double* mean, const double* stdv, double clip, const double* leg_zw,
                         int replicate, float* state, int32_t* node_idx, void* stream);

/* Replaces (batched over S env-steps): distribute_per_leg_reward / distribute_global_reward / distribute_contact_cost
 * (simulation_envs/quantruped_adaptor_multi_environment.py:160-203) and the GlobalCosts variant
 * (quantruped_fourDecentralizedController_GlobalCosts_environments.py:69-83), float64 arithmetic like numpy:
 *   fw_reward [S] (info['reward_forward']), actions [S][Ag][A] (unclipped policy outputs), cfrc_ext [S][NB][6] float64,
 *   contact_table [Ag][NB] float64 (weights of get_contact_force_indices, 0 = unused) -> rewards [S][Ag] float32.
 *   mode 0 per-leg, 1 per-leg with norm_reward, 2 global reward, 3 GlobalCosts.  Ag <= 8, NB <= 16. */
int ddrl_reward_split(const float* fw_reward, const float* actions, const double* cfrc_ext,
                      const double* contact_table, int64_t S, int Ag, int A, int NB, double ctrl_cost_weight,
                      double contact_cost_weight, int mode, float* rewards, void* stream);

/* Replaces: concatenate_actions (quantruped_adaptor_multi_environment.py:205-212) + RLlib clip_actions:
 *   env_actions [S][A_full][action_table[a][j]] = clip(actions [S][Ag][A], clip_lo, clip_hi); action_table [Ag][A] int32. */
int ddrl_concat_actions(const float* actions, const int32_t* action_table, int64_t S, int Ag, int A, int A_full,
                        float clip_lo, float clip_hi, float* env_actions, void* stream);

/* Replaces: compute_advantages + postprocess_ppo_gae (RLlib evaluation/postprocessing.py,
 * agents/ppo/ppo_tf_policy.py), selected by use_gae/gamma/lambda at
 * train_experiment_1_architecture_on_flat.py:119-120.  Reverse scan per column in float64:
 *   delta_t = r_t + gamma*(1-done_t)*V_{t+1} - V_t ;  A_t = delta_t + gamma*lambda*(1-done_t)*A_{t+1}
 *   rewards, values [P][T][C] float32; dones [T][C/cols_per_env] uint8 (shared by the policies and
 *   by the cols_per_env agent columns of one env); v_boot [P][C] float32 (V of the obs after step T-1)
 *   adv, vtarg [P][T][C] float32 (out);  moments [P][3] float64 (out): {count, sum(adv), sum(adv^2)}
 *   ws: ddrl_gae_ws_bytes(P, C). */
int64_t ddrl_gae_ws_bytes(int P, int64_t C);
int ddrl_gae(const float* rewards, const float* values, const uint8_t* dones, const float* v_boot,
             int P, int T, int64_t C, int cols_per_env, double gamma, double lambda, float* adv,
             float* vtarg, double* moments, void* ws, void* stream);

/* Replaces: StandardizeFields(["advantages"]) (RLlib execution/rollout_ops.py):
 *   adv <- (adv - mean) / max(1e-4, std)  per policy, population std, from moments[P][3]
 *   (moments may have been all-reduced across ranks first). In place. */
int ddrl_adv_standardize(float* adv, const double* moments, int P, int64_t R, void* stream);

/* Replaces: SampleBatch.shuffle() in TrainTFMultiGPU (RLlib execution/train_ops.py;
 * shuffle_sequences=true).  dst[p][i][:] = src[p][perm[p][i]][:] for a [P][R][W] float32 array. */
int ddrl_gather_rows(const float* src, const int32_t* perm, int P, int64_t R, int W, float* dst,
                     void* stream);

/* One minibatch of: model forward + PPOLoss + backward (no optimizer).
 * Replaces: one session.run of loss+grads in TrainTFMultiGPU for all P policies at once
 * (RLlib agents/ppo/ppo_tf_policy.py PPOLoss; DiagGaussian logp/kl/entropy).
 * Shapes: D <= 64, A <= 8, and D <= 60 for A = 8 (the kernel's shared memory exceeds 227 KB beyond that:
 * DDRL_E_UNSUPPORTED_SHAPE).
 * Batch arrays are [P][R][*] float32; the minibatch is rows [mb*MB, (mb+1)*MB) where
 *   mb = mb_perm[p][*step_ctr]          (device ints; lets one CUDA graph serve every step)
 *   kl_coeff [P] float32 (device),  hyper (host values): clip_param, vf_clip_param, vf_loss_coeff,
 *   entropy_coeff, inv_global_mb = 1 / (MB summed over all ranks).
 * Outputs (workspace, per CTA, reduced by ddrl_grad_reduce in fixed order -> deterministic):
 *   grad_part [P][G][NPs] float32 (NPs = NP rounded up to a multiple of 4),
 *   stat_part [P][G][DDRL_NSTAT] float64, G = ctas_per_policy
 *   stat sums: 0 sum(-surr) 1 sum(kl) 2 sum(vf) 3 sum(entropy) 4 sum(R) 5 sum(R^2)
 *              6 sum(R-v) 7 sum((R-v)^2)       (R = value_targets)
 * If ext_dlogits != NULL the loss is skipped and the row gradients are read from
 * ext_dlogits [P][R][2A] / ext_dvalue [P][R] (torch.autograd boundary of the ModelV2 classes). */
typedef struct {
    float clip_param, vf_clip_param, vf_loss_coeff, entropy_coeff, inv_global_mb;
} ddrl_ppo_hyper;

/* Optional fused tail of an SGD step (pass NULL to get the partials only): the train kernel itself then performs what
 * ddrl_grad_reduce + [gradient all-reduce] + ddrl_clip_adam would do — a barrier among the CTAs of each policy, the
 * fixed-order partial reduction (each CTA owns a slice of the parameters), at world > 1 an in-kernel all-reduce of the
 * slices over NVLink peer memory, the global-norm clip, TF1 Adam, the packed weight images, the beta powers and
 * *step_ctr — in ONE launch per step.  Requires ctas_per_policy * P <= number of SMs (all CTAs co-resident).
 * Device pointers:
 *   theta, m, v [P][NP]; beta_pow [P][2]; grad [P][NP] (out: reduced gradient); gnorm_out [P] or NULL;
 *   fcnet_img / fcnet_tc_img or NULL; step_stats [steps][P][DDRL_NSTAT] or NULL; step_ctr;
 *   barrier_ws: 4*P + 4 zero-initialised uint32 (counters re-armed by the kernel; [4P+1] = steps executed so far);
 *   sq_ws: P * ctas_per_policy zero-initialised 128-byte lines, first 64-bit word = {float ||g_slice||^2, uint32 step tag};
 *   status: device int or NULL, receives |= 64 when a bounded spin of the tail gave up (results then invalid);
 *   nsteps > 1: the launch runs that many consecutive optimizer steps (*step_ctr .. *step_ctr + nsteps - 1) as ONE
 *   persistent kernel — TMEM, barriers and the instruction stream stay warm, the launch gap disappears; the CTAs of a
 *   policy meet at a third barrier before they reload the updated weights.
 * Data parallel (world > 1; one process per GPU, every rank launches the same step with the same shapes):
 *   seq       device uint32, zero-initialised once, advanced by the kernel every step;
 *   peer_x[w] exchange buffer of rank w (peer-mapped, ddrl_peer_alloc/open; [rank] = the local one), zero-initialised:
 *             2 * world * P * ddrl_sgd_exchange_words(NP, ctas_per_policy) 64-bit words {float value, uint32 seq + 1}.
 * Every rank ends each step with bit-identical gradients (slices are summed in rank order) and weights. */
#define DDRL_MAX_RANKS 8
typedef struct {
    float *theta, *m, *v, *beta_pow, *grad, *gnorm_out, *fcnet_img;
    void* fcnet_tc_img;
    double* step_stats;
    int32_t* step_ctr;
    uint32_t* barrier_ws;
    float* sq_ws;
    float lr, beta1, beta2, eps, grad_clip;
    int32_t* status;          /* device int or NULL: OR-ed with 64 if a barrier / peer wait of the tail timed out */
    int32_t world, rank;
    uint32_t* seq;
    unsigned long long* peer_x[DDRL_MAX_RANKS];
    int32_t nsteps;           /* consecutive SGD steps per launch (0 or 1 = one); > 1 only ddrl_ppo_train_step_tc (ping-pong) */
    unsigned long long* ll_ws; /* NULL, or ddrl_sgd_ll_words(...) zero-initialised 64-bit words: the ping-pong kernel then hands partial
                                * gradients and updated weights between CTAs as self-validating {payload, step tag} words instead of
                                * barrier-protected arrays (one barrier-free tail per step; csrc/sgd_tail.cuh).  Must share the lifetime
                                * of barrier_ws (the tags are the step count kept there). */
    float* grad_acc;           /* NULL, or [P][NP rounded up to 4] ZERO-initialised floats: the ping-pong kernel then ADDS its per-CTA
                                * partial gradients into this one vector per policy (red.global.add.v4.f32 at L2) instead of writing
                                * ctas_per_policy partials that every slice owner re-reads — per step 45 KB instead of 1.4 MB read back per
                                * policy; the slice owner reads its slice once and zeroes it again.  The order of the float additions is
                                * then NOT fixed: results vary from run to run in the last bits (ranks of one run still end bit-identical,
                                * the exchange adds in rank order).  NULL keeps the fixed-order reduction (bit-reproducible). */
} ddrl_sgd_tail;

/* 64-bit words of ddrl_sgd_tail.ll_ws for P policies of an FCNet (D, A) stepped by ctas_per_policy CTAs each. */
int64_t ddrl_sgd_ll_words(int P, int ctas_per_policy, int D, int A);

/* 64-bit words per (rank, policy) in the exchange buffer: ctas_per_policy slices of ((NP + G - 1) / G rounded up to 4) */
int64_t ddrl_sgd_exchange_words(int NP, int ctas_per_policy);

/* Peer-mapped device memory for the in-kernel all-reduce (CUDA IPC; one process per GPU on one node).
 *   ddrl_peer_alloc: cudaMalloc + zero-fill `bytes` on the current device; *ptr = device pointer, handle64 = 64-byte
 *                    cudaIpcMemHandle_t to send to the other ranks (e.g. torch.distributed.all_gather_object);
 *   ddrl_peer_open:  map another rank's allocation into this process (enables peer access), *ptr = local alias;
 *   ddrl_peer_close / ddrl_peer_free: undo open / alloc. */
int ddrl_peer_alloc(int64_t bytes, void** ptr, void* handle64);
int ddrl_peer_open(const void* handle64, void** ptr);
int ddrl_peer_close(void* ptr);
int ddrl_peer_free(void* ptr);

int ddrl_ppo_train_step(const float* theta, const float* img, const float* obs, const float* actions,
                        const float* old_logits, const float* old_logp, const float* vf_preds,
                        const float* adv, const float* vtarg, const float* ext_dlogits,
                        const float* ext_dvalue, int P, int64_t R, int D, int A, int MB,
                        const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                        const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas_per_policy,
                        float* grad_part, double* stat_part, const ddrl_sgd_tail* tail, void* stream);

/* 1 if the SGD step accepts an FCNet of observation width D and action width A, else 0 (pure host):
 * tensor_cores = 0: ddrl_ppo_train_step (D <= 64, A <= 8, D <= 60 for A = 8);
 * tensor_cores = 1: ddrl_ppo_train_step_tc (D <= 63, A in {1,2,4,8}). */
int ddrl_fcnet_train_supported(int D, int A, int tensor_cores);

/* Stand-alone PPOLoss gradient w.r.t. the model outputs (same arithmetic as the fused kernel), for
 * models whose forward/backward are separate kernels (GraphNet):
 *   logits [P][R][2A], value [P][R] + batch arrays -> dlogits [P][R][2A], dvalue [P][R],
 *   stat_part [P][ctas][DDRL_NSTAT] float64 (reduce with ddrl_grad_reduce's stat path). */
int ddrl_ppo_loss_grad(const float* logits, const float* value, const float* actions,
                       const float* old_logits, const float* old_logp, const float* vf_preds,
                       const float* adv, const float* vtarg, int P, int64_t R, int A,
                       const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas, float* dlogits,
                       float* dvalue, double* stat_part, void* stream);

/* Fixed-order reduction of the per-CTA partials:
 *   grad [P][NP] float32 = sum_g grad_part[p][g][:NP]      (grad_part rows are NPs = (NP+3)&~3 floats apart)
 *   step_stats [*step_ctr][P][DDRL_NSTAT] float64 = sum_g stat_part[p][g][:]   (if step_stats) */
int ddrl_grad_reduce(const float* grad_part, const double* stat_part, int P, int G, int NP,
                     float* grad, double* step_stats, const int32_t* step_ctr, void* stream);

/* Replaces: tf.clip_by_global_norm(grads, grad_clip) (RLlib ppo_tf_policy.clip_gradients) and
 * tf.compat.v1.train.AdamOptimizer.apply_gradients, per policy:
 *   scale = clip / max(||g||_2, clip);  lr_t = lr*sqrt(1-b2^t)/(1-b1^t)
 *   m = b1*m + (1-b1)*g;  v = b2*v + (1-b2)*g^2;  theta -= lr_t*m/(sqrt(v)+eps);  b1^t,b2^t *= b1,b2
 *   grad [P][NP] (may have been NCCL-all-reduced), theta/m/v [P][NP],
 *   beta_pow [P][2] (device) = {b1^t, b2^t} to be used by THIS step (TF convention: initialised to
 *   {b1, b2}, multiplied after the update), gnorm_out [P] or NULL,
 *   sync_ws: one zero-initialised int32 (device) used as an arrival ticket; the last CTA to finish
 *   multiplies the beta powers, increments *step_ctr (if not NULL) and re-zeroes the ticket.
 *   fcnet_img / fcnet_tc_img (or NULL): packed FP32 image [P][ddrl_fcnet_image_floats(img_D, img_A)] and tensor-core
 *   image [P][ddrl_fcnet_tc_image_bytes(img_D, img_A)] of the FCNet weights, updated in step with theta. */
int ddrl_clip_adam(float* theta, float* m, float* v, float* beta_pow, const float* grad, int P,
                   int NP, float lr, float beta1, float beta2, float eps, float grad_clip,
                   float* gnorm_out, int32_t* step_ctr, int32_t* sync_ws, float* fcnet_img,
                   void* fcnet_tc_img, int img_D, int img_A, void* stream);

/* ---------------------------------------------------------------------------------------------
 * GraphNet (models/graph_net.py:10-45) + actor/critic wrapper
 * (models/shared_graphnet_glorot_uniform_init.py:21-58).  Parameter layout per GraphNet(O), Keras
 * variable order: state_enc/kernel[4,19*64] state_enc/bias[19*64] msg_transform/kernel[64,64]
 * node_update/kernel[64,64] linear_out/kernel[64,O] linear_out/bias[O]; the wrapper stores
 * theta = [actor GraphNet(2A) | critic GraphNet(1)].
 *   node_idx [B] int32, state [B][4][23] float32, adj [B][4][4] float32 (adj[s][r]!=0: edge s->r)
 *   -> logits [B][2A], value [B].
 * ------------------------------------------------------------------------------------------- */
int ddrl_graphnet_num_params(int num_outputs);
int ddrl_graphnet_forward(const float* theta, const int32_t* node_idx, const float* state,
                          const float* adj, int64_t B, int A, float* logits, float* value,
                          void* stream);
/* Forward schedule (A/B timing and tests) of ddrl_graphnet_forward: 0 = one row per CTA, 1 = one row per warp with the
 * weights in shared memory, -1 = library default (overridable by the environment variable DDRL_GN_FWD_VARIANT=0|1).  Same
 * results up to the FP32 summation order.  ddrl_graphnet_act always runs the row-per-warp schedule. */
int ddrl_graphnet_set_variant(int variant);
/* GraphNet inference + DiagGaussian sampling in ONE launch (the sampler-side call of the shared graph policy):
 *   theta, node_idx [B], state [B][4][23], adj [B][4][4] as in ddrl_graphnet_forward, eps [B][A] (all required)
 *   -> logits [B][2A], value [B], action [B][A] = mean + exp(log_std) * eps, logp [B] (the logp of that action).
 * logits / value are bit-identical to ddrl_graphnet_forward under forward schedule 1 (one warp per row); action / logp
 * are bit-identical to ddrl_dg_sample applied to those logits. */
int ddrl_graphnet_act(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                      const float* eps, int64_t B, int A, float* logits, float* value, float* action, float* logp,
                      void* stream);
/* Backward of the wrapper w.r.t. theta from dlogits [B][2A], dvalue [B]:
 *   grad_part [G][NPs] per-CTA partials, NPs = (NP+3)&~3 (reduce with ddrl_grad_reduce(P=1)); G = ctas. */
int ddrl_graphnet_backward(const float* theta, const int32_t* node_idx, const float* state,
                           const float* adj, const float* dlogits, const float* dvalue, int64_t B,
                           int A, int ctas, float* grad_part, void* stream);

/* One SGD step of the GraphNet wrapper in two launches (opt-in alternative to ddrl_graphnet_forward + ddrl_ppo_loss_grad +
 * ddrl_graphnet_backward; same arithmetic): (1) one warp per row: forward, the row's PPOLoss gradient w.r.t. this net's
 * outputs (policy part for the actor, value part for the critic; RLlib ppo_tf_policy.PPOLoss) and the backward down to the
 * layer inputs, leaving a 2.1 KB record per (net, row) in `ws`; (2) thread-owned register accumulation of the weight
 * gradients over the rows of each CTA.
 *   theta, node_idx [B], state [B][4][23], adj [B][4][4] as in ddrl_graphnet_forward; actions [B][A], old_logits [B][2A],
 *   old_logp / vf_preds / adv / vtarg [B]; kl_coeff: device float; ws: ddrl_graphnet_train_ws_bytes(B) bytes;
 *   grad_part [ctas][NPs] per-CTA partials like ddrl_graphnet_backward (reduce with ddrl_grad_reduce(P=1));
 *   stat_part [ddrl_graphnet_train_stat_parts(B)][DDRL_NSTAT] float64 partial sums (actor CTAs fill the policy entries,
 *   critic CTAs the value entries; sum them all). */
int64_t ddrl_graphnet_train_ws_bytes(int64_t B);
int ddrl_graphnet_train_stat_parts(int64_t B);
int ddrl_graphnet_train_step(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                             const float* actions, const float* old_logits, const float* old_logp,
                             const float* vf_preds, const float* adv, const float* vtarg, int64_t B, int A,
                             const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas, void* ws,
                             float* grad_part, double* stat_part, void* stream);

/* GraphNet SGD steps on tensor cores (csrc/graphnet_tc.cu): ONE persistent kernel per launch runs, for every optimizer step,
 * forward + PPOLoss + backward of the actor / critic wrapper and (with `tail`) the fused gradient reduce + [NVLink all-reduce]
 * + clip + TF1 Adam.  The hyper-network leg encoder (1216 tanh per (row, node) pair; not a contraction) runs on the FMA + MUFU
 * pipes with thread-owned columns; the MPNN (msg_transform / node_update), the linear head, their transposes and the
 * K = rows weight-gradient GEMMs run on tcgen05 with fp16 hi/lo split operands (3 products, FP32 accumulation in TMEM).
 *   batch arrays as ddrl_graphnet_train_step but for ALL R rows; step k of the launch trains rows
 *   [mb * MB, mb * MB + MB) with mb = mb_perm[*step_ctr + k] (mb_perm NULL: mb = step);
 *   grid = 2 x ctas_per_net CTAs (all co-resident: 2 * ctas_per_net <= #SMs);
 *   grad_part [ctas_per_net][NPs] (row i: actor half from actor CTA i, critic half from critic CTA i; reduce with
 *   ddrl_grad_reduce(P = 1, G = ctas_per_net) when tail == NULL); stat_part [2 * ctas_per_net][DDRL_NSTAT] float64,
 *   ZERO-INITIALISED by the caller (rows >= ctas_per_net are never written);
 *   tail: ddrl_sgd_tail for P = 1, NP = ddrl_graphnet_num_params(2A), 2 * ctas_per_net CTAs (sq_ws / exchange buffers sized
 *   for that CTA count), fcnet_img / fcnet_tc_img / ll_ws NULL; tail->nsteps consecutive steps per launch;
 *   status: device int or NULL (1 MMA wait timed out, 8 / 16 fp16 range of the loss gradients exceeded, 64 tail wait). */
int ddrl_graphnet_train_step_tc(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                                const float* actions, const float* old_logits, const float* old_logp,
                                const float* vf_preds, const float* adv, const float* vtarg, int64_t R, int A, int MB,
                                const int32_t* mb_perm, const int32_t* step_ctr, const float* kl_coeff,
                                const ddrl_ppo_hyper* hyper, int ctas_per_net, float* grad_part, double* stat_part,
                                int* status, const ddrl_sgd_tail* tail, void* stream);

/* GCN layer (models/gcn.py:7-37, graph_ops.adj_norm models/graph_ops.py:13-21):
 *   y = act((D^-1 A) X W + b), X [B][4][F], A [B][4][4], W [F][U], b [U] or NULL, act: 0 none 1 tanh */
int ddrl_gcn_forward(const float* x, const float* adj, const float* W, const float* b, int64_t B,
                     int F, int U, int act, float* y, void* stream);

/* Graph-layer variants the reference carries but does not wire into a model (SURVEY.md §8-f N1),
 * 4-node graphs: X [B][4][F], A [B][4][4] (adj[s][r] != 0 => edge s -> r), F, U <= 64, act: 0 none, 1 tanh.
 *   MPNN2 (models/gcn.py:96-150):  e = [x_s, x_r] W_msg (W_msg [2F][U]);  m_r = mean of incoming e (0 if none);
 *                                   y = act([x, m] W_upd + b)  (W_upd [F+U][U], b [U] or NULL)
 *   GAT1  (models/gcn.py:153-206): self loops added; x' = x W_pre (W_pre [F][U]); a = leaky_relu_0.2(w_att . [x'_s, x'_r])
 *                                   (w_att [2U]); softmax of a over the edges of each receiver; y_s = act(sum_r Att[s][r] x'_r + b)
 *   symm_norm (models/graph_ops.py:3-11): D^-1/2 A D^-1/2 for A [B][N][N], N <= 64 (zero degree -> NaN like the reference)
 *   segment_softmax (models/graph_ops.py:23-26): out = exp(data) / segment_sum(exp(data)); data [E][C], segment_ids [E]
 *       int32 in [0, num_segments); sums_ws [num_segments][C] floats and bad_id (device int: 1 if an id was out of
 *       range) are scratch; sums use float atomics (order-dependent in the last bits). */
int ddrl_mpnn2_forward(const float* x, const float* adj, const float* W_msg, const float* W_upd, const float* b,
                       int64_t B, int F, int U, int act, float* y, void* stream);
int ddrl_gat1_forward(const float* x, const float* adj, const float* W_pre, const float* w_att, const float* b,
                      int64_t B, int F, int U, int act, float* y, void* stream);
/* Backward of the two layers (tf.gradients through models/gcn.py:96-206): dy [B][4][U] -> dx [B][4][F] (or NULL) and per-CTA
 * partial weight gradients grad_part [ctas][NPs], NPs = (NP + 3) & ~3, flat order MPNN2 [W_msg (2F x U) | W_upd ((F + U) x U) |
 * b (U)], GAT1 [W_pre (F x U) | w_att (2U) | b (U)] (the b entries are written even when b == NULL); reduce with
 * ddrl_grad_reduce(P = 1, G = ctas).  Fixed order, no atomics. */
int ddrl_mpnn2_backward(const float* x, const float* adj, const float* W_msg, const float* W_upd, const float* b,
                        const float* dy, int64_t B, int F, int U, int act, int ctas, float* dx, float* grad_part, void* stream);
int ddrl_gat1_backward(const float* x, const float* adj, const float* W_pre, const float* w_att, const float* b,
                       const float* dy, int64_t B, int F, int U, int act, int ctas, float* dx, float* grad_part, void* stream);
int ddrl_symm_norm(const float* adj, int64_t B, int N, float* out, void* stream);
int ddrl_segment_softmax(const float* data, const int32_t* segment_ids, int64_t E, int C, int64_t num_segments,
                         float* sums_ws, int* bad_id, float* out, void* stream);

/* DiagGaussian sample + logp (RLlib models/tf/tf_action_dist.py DiagGaussian._build_sample_op / logp)
 * for models without a fused epilogue: action = mean + exp(log_std)*eps, logp(action).
 *   logits [R][2A], eps [R][A] -> action [R][A], logp [R]. */
int ddrl_dg_sample(const float* logits, const float* eps, int64_t R, int A, float* action, float* logp,
                   void* stream);

/* LegCoupling (models/coupling_net_glorot_uniform_init.py:11-30,135):
 *   logits[b][j] *= (j < 2 ? coupling[node_id[b]][j] : 1)      in place; coupling [4][2]. */
int ddrl_leg_coupling(float* logits, const int32_t* node_id, const float* coupling, int64_t B,
                      int W, void* stream);
/* Backward of the layer (the table is a TRAINABLE tf.Variable registered with the model,
 * models/coupling_net_glorot_uniform_init.py:20-21,160-161):
 *   dcoupling[n][j] = sum_{b: node_id[b] == n} dout[b][j] * logits_pre[b][j]   (j < 2; [4][2], overwritten)
 *   dout[b][j]     *= coupling[node_id[b]][j]                                   (in place -> gradient w.r.t. logits_pre)
 * Fixed-order reduction (one block, float64 partial sums): bit-reproducible. */
int ddrl_leg_coupling_backward(float* dout, const float* logits_pre, const int32_t* node_id,
                               const float* coupling, int64_t B, int W, float* dcoupling, void* stream);

/* Optional FCNet layouts (`vf_share_layers`, `free_log_std`; models/fcnet_glorot_uniform_init.py:30-36,85-113) on the two-branch
 * kernels.  The kernels' parameter vector [NPk] is an index-select of the model's variables [NPm]:
 *   ddrl_param_expand: theta_kernel[p][i] = map[i] in [0, NPm) ? theta_model[p][map[i]] : 0      (map [NPk] int32)
 *   ddrl_grad_tie:     grad_model[p][j] = sum of grad_kernel[p][inv[j][k]], k = 0, 1 (inv [NPm][2] int32, -1 = none; fixed
 *                      order) — the gradients of tied copies add up, gradients of constant entries are dropped. */
int ddrl_param_expand(const float* theta_model, const int32_t* map, int P, int NPm, int NPk, float* theta_kernel, void* stream);
int ddrl_grad_tie(const float* grad_kernel, const int32_t* inv, int P, int NPm, int NPk, float* grad_model, void* stream);

/* Tensor-core variant of ddrl_ppo_train_step (PPO path only): every GEMM of the fused forward + loss + backward
 * runs on tcgen05 (kind::f16, FP32 accumulation in TMEM) with FP32 operands split into fp16 (hi, lo) pairs and
 * three products per GEMM, which keeps the 1e-5 parity bar.  Same batch arrays, minibatch selection, outputs
 * (grad_part [P][G][NPs], stat_part) and semantics as ddrl_ppo_train_step; the weights come from a tensor-core
 * image tc_img [P][ddrl_fcnet_tc_image_bytes(D, A)] built by ddrl_fcnet_tc_pack (or kept in step by
 * ddrl_clip_adam).  D <= 63, A in {1,2,4,8} (ddrl_fcnet_tc_image_bytes / ddrl_fcnet_tc_pack refuse other shapes).  *status (device int, may be NULL) receives OR-ed flags: 1 = an MMA
 * completion wait timed out; 64 = a fused-tail barrier timed out; 2/4/8/16/32 = fp16 overflow (clamped) while splitting x / activations / dl / dz2 / dz1 —
 * the result is then unreliable and the step should be redone with ddrl_ppo_train_step. */
int ddrl_fcnet_tc_image_bytes(int D, int A);
/* Inference on the tensor cores: same contract as ddrl_fcnet_forward (filter normalise prologue, logits / value,
 * DiagGaussian sample + logp epilogue) with the GEMMs on tcgen05 (fp16 hi/lo split, ~3e-6 relative); weights from the
 * tensor-core image.  Shapes the ping-pong kernel covers: D <= 47, A in {1,2,4,8}.  Any of obs_out / logits / value /
 * eps (+ action, logp) may be NULL. */
int ddrl_fcnet_forward_tc(const void* tc_img, const float* obs, const double* norm, float clip, int P, int64_t R,
                          int D, int A, float* obs_out, float* logits, float* value, const float* eps,
                          float* action, float* logp, int* status, void* stream);
/* Two schedules of the same arithmetic exist: 1 = branch-sequential (any D <= 63), 2 = "ping-pong" (both branches
 * resident, the tensor core runs one branch while the CTA runs the other's epilogue; D <= 47, A in {1,2,4,8}).
 * 0 (default) picks ping-pong whenever the shape allows it.  Process-wide; meant for tests and A/B timing. */
int ddrl_tc_set_variant(int variant);
/* 1 if ddrl_ppo_train_step_tc will use the ping-pong kernel for (D, A) under the current variant setting (the kernel that
 * accepts ddrl_sgd_tail.nsteps > 1), else 0. */
int ddrl_tc_pingpong_eligible(int D, int A);
/* Thread-block clusters of the ping-pong kernel: the CTAs of a cluster add their partial gradients over distributed
 * shared memory, so one partial per CLUSTER (not per CTA) goes through L2.  1 (default) = no clusters — on the bench
 * workload the per-step time is set by the three CTA-group barriers, not by the partial traffic, and clusters of 4 measured
 * 5 % slower; -1 = the largest of 16, 8, 4, 2 that divides ctas_per_policy and keeps every cluster co-resident; 2/4/8/16 =
 * that size.  ddrl_tc_last_cluster() returns the size the most recent launch used. */
int ddrl_tc_set_cluster(int cluster_size);
int ddrl_tc_last_cluster(void);
/* Diagnostic: when non-NULL (device int64[64 + 8 * #CTAs]), thread 0 of CTA (0, 0) of the ping-pong kernel stores clock64()
 * at its phase boundaries (index = phase number) and thread 0 of EVERY CTA stores %globaltimer at 8 points of the step
 * ([64 + 8 * cta + k]) — in-kernel timing without a profiler.  NULL switches it off. */
int ddrl_tc_set_debug_clock(void* device_int64x64);
int ddrl_fcnet_tc_pack(const float* theta, int P, int D, int A, void* tc_img, void* stream);
int ddrl_ppo_train_step_tc(const void* tc_img, const float* obs, const float* actions,
                           const float* old_logits, const float* old_logp, const float* vf_preds,
                           const float* adv, const float* vtarg, int P, int64_t R, int D, int A, int MB,
                           const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                           const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas_per_policy,
                           float* grad_part, double* stat_part, int* status, const ddrl_sgd_tail* tail,
                           void* stream);

/* Leg-coupled SGD steps: the policy of QuantrupedMultiEnv_SharedDecentralLegID, model "cup" = FCNet + LegCoupling
 * (models/__init__.py:7-13, models/coupling_net_glorot_uniform_init.py:11-30,135; ModelV2 class
 * FullyConnectedNetwork_Coupling_GlorotUniformInitializer).  Same batch arrays, minibatch selection and partial / stat
 * outputs as ddrl_ppo_train_step / ddrl_ppo_train_step_tc, with:
 *   logits[r][i] = pre[r][i] * coupling[node_id[r]][i]   (i < 2: the mean logits; the log-std half and the value are not scaled)
 *   the PPO loss taken of the coupled logits (old_logits are the coupled logits the actions were sampled from);
 *   d pre[r][i] = d logits[r][i] * coupling[node_id[r]][i];  d coupling[n][i] = sum_{r: node_id[r] = n} d logits[r][i] * pre[r][i]
 *   node_id [P][R] int32 in 0..3 (the agent's position in agent_names: FL, HL, HR, FR), in the batch's row order;
 *   theta [P][NP + 8]: the 12 FCNet variables in checkpoint order (NP = ddrl_fcnet_num_params(D, 2)), then leg_coupling [4][2]
 *     row-major — the registration order of the ModelV2 class; the coupling table is read from it every step;
 *   grad_part [P][G][(NP + 8 + 3) & ~3]; the fused tail is REQUIRED (tail->theta == theta, m / v / grad [P][NP + 8]) and
 *     clips + steps all NP + 8 parameters (the packed weight images get the first NP);
 *   A = 2 and P = 1 only (the reference builds this model as one shared policy; a wider action or several policies return
 *   DDRL_E_BADARG); no LL tail, no thread-block clusters (DDRL_E_BADARG).
 * A node id outside 0..3 read on the device sets *status |= DDRL_STATUS_BAD_NODE (the row is then coupled as node id & 3).
 * ddrl_ppo_train_step_coupled is the FP32 step (nsteps <= 1; *tail->status, REQUIRED, receives the flag; weights from the
 * packed image img, ddrl_fcnet_pack of the first NP entries); ddrl_ppo_train_step_tc_coupled the ping-pong tensor-core step
 * (tail->nsteps consecutive steps per launch; D in {19, 20}; status REQUIRED; weights from the tensor-core image tc_img,
 * ddrl_fcnet_tc_pack of the first NP).  A NULL status is rejected with DDRL_E_BADARG, so a bad node id cannot go unreported. */
#define DDRL_STATUS_BAD_NODE 128
int ddrl_ppo_train_step_coupled(const float* theta, const float* img, const int32_t* node_id, const float* obs,
                                const float* actions, const float* old_logits, const float* old_logp, const float* vf_preds,
                                const float* adv, const float* vtarg, int P, int64_t R, int D, int A, int MB,
                                const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr, const float* kl_coeff,
                                const ddrl_ppo_hyper* hyper, int ctas_per_policy, float* grad_part, double* stat_part,
                                const ddrl_sgd_tail* tail, void* stream);
int ddrl_ppo_train_step_tc_coupled(const void* tc_img, const float* theta, const int32_t* node_id, const float* obs,
                                   const float* actions, const float* old_logits, const float* old_logp,
                                   const float* vf_preds, const float* adv, const float* vtarg, int P, int64_t R, int D,
                                   int A, int MB, const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                                   const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas_per_policy,
                                   float* grad_part, double* stat_part, int* status, const ddrl_sgd_tail* tail,
                                   void* stream);
/* Inference of the leg-coupled policy in ONE launch (the sampler-side call and the rollout forward of SharedDecentralLegID):
 * the contract of ddrl_fcnet_forward / ddrl_fcnet_forward_tc (filter prologue, obs_out, logits, value, DiagGaussian sample
 * epilogue; any of obs_out / logits / value / eps (+ action, logp) may be NULL) with LegCoupling applied to the logits:
 *   node_id [P][R] int32 in 0..3, coupling [4][2] (the table, theta[NP .. NP + 8) of the coupled learner);
 *   logits[r][i] = pre[r][i] * coupling[node_id[r]][i] for i < 2 (one rounding; the log-std half and value unchanged), and
 *   action / logp are drawn from that coupled DiagGaussian.
 * Bit-identical to ddrl_fcnet_forward (resp. ddrl_fcnet_forward_tc) -> ddrl_leg_coupling -> ddrl_dg_sample on the same
 * inputs.  A node id outside 0..3 sets *status |= DDRL_STATUS_BAD_NODE (the row is then coupled as node id & 3); status is
 * REQUIRED.  A = 2 and P = 1 only (DDRL_E_BADARG otherwise, as for the null pointers and R < 0); R = 0 does nothing.
 * ddrl_fcnet_forward_coupled is the FP32 kernel (weights from theta [P][NP] or the packed image img); the tensor-core entry
 * takes the tensor-core image and is instantiated for D in {19, 20} (DDRL_E_UNSUPPORTED_SHAPE otherwise). */
int ddrl_fcnet_forward_coupled(const float* theta, const float* img, const int32_t* node_id, const float* coupling,
                               const float* obs, const double* norm, float clip, int P, int64_t R, int D, int A,
                               float* obs_out, float* logits, float* value, const float* eps, float* action, float* logp,
                               int* status, void* stream);
int ddrl_fcnet_forward_tc_coupled(const void* tc_img, const int32_t* node_id, const float* coupling, const float* obs,
                                  const double* norm, float clip, int P, int64_t R, int D, int A, float* obs_out,
                                  float* logits, float* value, const float* eps, float* action, float* logp, int* status,
                                  void* stream);

/* Diagnostic: one tcgen05 (UMMA) GEMM through TMEM with the chunked shared-memory operand layout the tensor-core
 * training step uses (csrc/umma.cuh): D[m][n] = sum_k A(m,k) B(n,k), m < M (64 or 128), A(m,k) = A[m][k] (a_mn = 0, K-major) or
 * A[k][m] (a_mn = 1, MN-major view); B alike; split != 0 -> fp16 (hi, lo) operand split with three products.
 * A [ra][ca], B [rb][cb] float32 device arrays; D [128][N] = the raw TMEM lanes 0..127 x N columns (for M = 64 the
 * accumulator rows occupy a subset of the lanes); *status (device int) = 0 ok, 1 = MMA completion timed out. */
int ddrl_umma_selftest(const float* A, int ra, int ca, const float* B, int rb, int cb, int M, int N, int K,
                       int a_mn, int b_mn, int split, float* D, int* status, void* stream);

/* Diagnostic micro-benchmark: `reps` x `ksteps` back-to-back tcgen05.mma kind::f16 (M x N x 16, operands in the chunked
 * layout, a_mn / b_mn = MN-major views) issued by one thread; cycles2 (device int64[2]) = {issue loop, issue + completion}. */
int ddrl_umma_bench(int M, int N, int a_mn, int b_mn, int reps, int ksteps, void* cycles2, int* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDRL_B200_H */
