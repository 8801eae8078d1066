/*
 * simstep.h — C ABI of libsimstep.so: the B200 (sm_100a) implementation of the
 * batched learned-dynamics environment step of gym-simenv / MILO.
 *
 * Every entry point below replaces one call on the reference's hot path.  The
 * citations are paths under the reference tree (file:line):
 *
 *   SE  = gym-simenv/gym_simenv/envs/sim_env.py
 *   DYN = milo/milo/dynamics.py
 *   LC  = milo/milo/linear_cost.py
 *   SI  = deepmimic/deepmimic/DeepMimicCore/scenes/SceneImitate.cpp
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary.
 *   - pointers named *_dev are CUDA device pointers owned by the caller,
 *     pointers named *_host are host pointers, read during the call only.
 *   - `stream` is a cudaStream_t passed as void*; all device work is enqueued
 *     on it and the call returns without synchronising unless stated.
 *   - every function returns 0 on success, a negative SIMSTEP_E* code on
 *     failure; simstep_last_error() gives the message.  Nothing throws.
 *   - a handle is bound to the CUDA device that was current at create time and
 *     is not thread-safe: one handle per GPU per thread.
 *   - all matrices are row-major fp32 and dense unless a pitch is given.
 */
#ifndef SIMSTEP_H_
#define SIMSTEP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIMSTEP_ABI_VERSION 1

#define SIMSTEP_OK 0
#define SIMSTEP_EINVAL (-1)   /* bad argument / wrong call order            */
#define SIMSTEP_ECUDA (-2)    /* a CUDA runtime or driver call failed        */
#define SIMSTEP_ENODEV (-3)   /* no sm_100 device                           */
#define SIMSTEP_ENOMEM (-4)   /* workspace allocation failed                */

#define SIMSTEP_MAX_HIDDEN 8
#define SIMSTEP_MAX_BODIES 32
#define SIMSTEP_MAX_JOINTS 32

/* operand formats of the tensor-core GEMMs (fp32 accumulate in TMEM) */
#define SIMSTEP_PREC_TF32 0   /* 10-bit mantissa, 8-bit exponent: any range    */
#define SIMSTEP_PREC_FP16 1   /* 10-bit mantissa, 5-bit exponent, saturating: twice the tf32 rate; the host mirror's default */
#define SIMSTEP_PREC_BF16 2   /* 7-bit mantissa, 8-bit exponent              */

#define SIMSTEP_ACT_RELU 0
#define SIMSTEP_ACT_TANH 1

#define SIMSTEP_SHAPE_SPHERE 0
#define SIMSTEP_SHAPE_CAPSULE 1
#define SIMSTEP_SHAPE_BOX 2   /* ignored, as SE:238-244 does */

typedef struct simstep_handle simstep_handle;

/* Shape of the dynamics ensemble: the ctor arguments of DynamicsEnsemble
 * (DYN:19-80) and BasicMLP (DYN:394-420) that matter for inference. */
typedef struct simstep_config {
  int32_t abi_version;      /* SIMSTEP_ABI_VERSION                           */
  int32_t state_dim;        /* S, 226 for humanoid3d                         */
  int32_t action_dim;       /* A, 28                                         */
  int32_t n_models;         /* N ensemble members (DYN:26)                   */
  int32_t n_hidden;         /* number of hidden layers                       */
  int32_t hidden[SIMSTEP_MAX_HIDDEN]; /* hidden_sizes (DYN:28)               */
  int32_t dense_connect;    /* DYN:30, DYN:414-419                           */
  int32_t activation;       /* SIMSTEP_ACT_* (DYN:31, DYN:410)               */
  int32_t transform;        /* DYN:32: normalise in / un-normalise out       */
  int32_t precision;        /* SIMSTEP_PREC_*                                */
  int32_t max_chunk_envs;   /* workspace rows per pass; 0 = default          */
  int32_t reserved[7];
} simstep_config;

/* Termination model of SimEnv.is_done (SE:164-268). */
typedef struct simstep_termination {
  int32_t horizon;               /* SE:28, SE:170                            */
  int32_t enable_velocity_check; /* SE:27, SE:172                            */
  int32_t vel_offset;            /* deepmimic.get_vel_offset(), 136          */
  float vel_threshold;           /* SE:259, 100                              */
  float vel_divisor;             /* sampling_rate if RecordVelAsPos else 1   */
  int32_t record_all_world;      /* SE:181, SE:227                           */
  int32_t record_world_root_pos; /* SE:181, SE:227                           */
  int32_t n_bodies;              /* len(fall_contact_bodies), SE:102         */
  int32_t body_offset[SIMSTEP_MAX_BODIES]; /* (pos+rot dim)*id + 1, SE:103   */
  int32_t body_shape[SIMSTEP_MAX_BODIES];  /* SIMSTEP_SHAPE_*                */
  float body_param0[SIMSTEP_MAX_BODIES];   /* diameter, SE:188, SE:201       */
  float body_param1[SIMSTEP_MAX_BODIES];   /* cylinder height, SE:202        */
  int32_t pos_dim;               /* 3, SE:99                                 */
} simstep_termination;

/* ---- lifetime ----------------------------------------------------------- */

int simstep_abi_version(void);
/* Message of the last failure on this handle (or of the last failed create
 * when h is NULL).  The pointer stays valid until the next call. */
const char* simstep_last_error(const simstep_handle* h);

int simstep_create(const simstep_config* cfg, simstep_handle** out);
int simstep_destroy(simstep_handle* h);

/* Packed-operand geometry, for callers that size buffers and for tests. */
int simstep_query(const simstep_handle* h, int32_t* n_layers, int32_t* layer_in /*[n_layers]*/,
                  int32_t* layer_out /*[n_layers]*/, int64_t* chunk_envs, int64_t* workspace_bytes);

/* ---- parameters --------------------------------------------------------- */

/* Replaces DynamicsEnsemble.load_ensemble / DynamicsModel.load (DYN:118-131,
 * DYN:380-386): weights_host[m*n_layers+l] is fc_layers.l.weight of member m
 * ([out,in] row-major, in = BasicMLP's concat width), biases_host likewise.
 * transforms_host = {state_mean, state_scale, action_mean, action_scale,
 * diff_mean, diff_scale} (DS:23-43), ignored when cfg.transform == 0. */
int simstep_load_ensemble(simstep_handle* h, const float* const* weights_host,
                          const float* const* biases_host, const float* const* transforms_host);

int simstep_set_termination(simstep_handle* h, const simstep_termination* t);

/* Number of normalised inputs (s - mean) / scale whose magnitude exceeded the fp16 range (65 504) since the last
 * reset - only counted for SIMSTEP_PREC_FP16 handles, which saturate there while the fp32 reference carries on
 * (DYN:225-227 divides by a scale that DS:35-40 lets be 1e-8 for a constant dataset column).  Synchronises with
 * the device.  A non-zero count means: use SIMSTEP_PREC_TF32 for this data. */
int simstep_saturation_count(simstep_handle* h, int64_t* count_out, int32_t reset);

/* How many launches the ensemble forward pass (DYN:422-433 for every member, all layers) takes for a pass of
 * n_envs rows on this handle: 1 when the column-fused kernel runs (a CTA pair carries a (member, 256-row env tile)
 * through every layer, activations handed on through L2 - used while the packed weights plus one unit's activation
 * rows per CTA pair fit the L2), n_hidden + 1 when every layer is a grouped launch of its own.  No reference
 * counterpart (BasicMLP.forward is one Python loop, DYN:427-432); reported by bench.py beside the timings. */
int simstep_forward_launches(const simstep_handle* h, int64_t n_envs, int32_t* launches_out);

/* Out-of-bounds check of the handle's workspaces (compute-sanitizer is not available where the GPU tests run): with
 * SIMSTEP_DEBUG_GUARDS=1 in the environment at simstep_create every workspace buffer (normalised inputs, activations,
 * member deltas, cost operand rows, partial dots) is allocated between two 64 KB guard zones filled with 0xA5.
 * buffers_out = guarded buffers currently allocated (0 when the switch is off), bad_bytes_out = guard bytes that
 * have been overwritten.  Synchronises with the device.  No reference counterpart. */
int simstep_debug_check_guards(simstep_handle* h, int64_t* buffers_out, int64_t* bad_bytes_out);

/* The work-item schedule of the column-fused forward kernel for m_tiles 256-row env tiles and `groups` members on a
 * device with sm_count SMs, computed on the HOST with the kernel's own code (no handle, no GPU): CTA pairs used, whole
 * rounds that take an env tile's members in sequence, units of the last partial round shared by two pairs, and per pair
 * the list of (unit, role) items - unit = env_tile * groups + member, role -1 = the whole unit, 0 / 1 = one half of a
 * shared unit - terminated by (-1, -1); items_out is [pairs][max_items][2].  Test hook for the scheduling arithmetic. */
int simstep_debug_chain_schedule(int32_t m_tiles, int32_t groups, int32_t sm_count, int32_t max_items,
                                 int32_t* pairs_out, int32_t* seq_rounds_out, int32_t* tail_units_out,
                                 int32_t* items_out);

/* Replaces the rff layer of RBFLinearCost (LC:53-55): weight_host [D,in_dim],
 * bias_host [D].  in_dim must be S (input_type 's'), 2S ('ss'), S+A ('sa') or
 * 2S+A ('sas').  split != 0 keeps ~21 mantissa bits of the pre-activation by
 * running the GEMM on hi/lo operand pairs. */
int simstep_load_rff(simstep_handle* h, int32_t feature_dim, int32_t in_dim,
                     const float* weight_host, const float* bias_host, int32_t split);

/* Switches the hi/lo evaluation of a layer loaded with split != 0 off (one
 * product, a third of the tensor work, half of the operand-row bytes) or back
 * on, without re-uploading anything.  The pre-activation W_r x + b_r feeds a
 * cosine (LC:64-71), so what matters is its ABSOLUTE error: callers measure it
 * on their own data (amp_extensions_b200.RBFLinearCost does in fit_cost) and
 * keep the split only where plain operands would miss the 1e-3 budget. */
int simstep_set_rff_split(simstep_handle* h, int32_t split);

/* ---- ensemble forward --------------------------------------------------- */

/* DynamicsModel.forward(state, action, unnormalize_out=True) for ALL members
 * at once (DYN:216-233, DYN:422-433): delta_dev[m][e][:] is member m's
 * predicted state difference, layout [N][E][S]. */
int simstep_forward(simstep_handle* h, const float* state_dev, const float* action_dev, int64_t n_envs,
                    float* delta_dev, void* stream);

/* DynamicsEnsemble.compute_discrepancy (DYN:134-143): disc_dev[e] =
 * max_{i<j} ||delta_i - delta_j||_2. */
int simstep_discrepancy(simstep_handle* h, const float* state_dev, const float* action_dev, int64_t n_envs,
                        float* disc_dev, void* stream);

/* ---- the env step ------------------------------------------------------- */

/* Batched SimEnv.step + is_done (SE:140-173) with the discrepancy of
 * DYN:134-143 taken from the same forward pass.
 *   member_dev[e]    active member of env e (SE:282-283), int32
 *   num_steps_dev[e] step counter (SE:153), incremented in place, int32
 *   next_state_dev   [E][S]; may alias state_dev (SE:158 is in place)
 *   disc_dev         [E] or NULL
 *   done_dev         [E] uint8 or NULL
 */
int simstep_step(simstep_handle* h, const float* state_dev, const float* action_dev, const int32_t* member_dev,
                 int32_t* num_steps_dev, int64_t n_envs, float* next_state_dev, float* disc_dev, uint8_t* done_dev,
                 void* stream);

/* simstep_step followed by RBFLinearCost.get_bonus_costs (LC:111-152) on the
 * same rows, input_type taken from simstep_load_rff:
 *   w_dev [D]       cost weights (LC:91)
 *   cost = (1-lambda_b)*clamp(phi.w, c_min, c_max) - lambda_b*min(disc/threshold,1)*c_min
 *   cost_dev, ipm_dev, bonus_dev: [E] each, any may be NULL (bonus is the
 *   weighted bonus, LC:144).  clamp_cost == 0 reproduces cost_range=None
 *   (LC:137-138, LC:103). */
int simstep_step_cost(simstep_handle* h, const float* state_dev, const float* action_dev,
                      const int32_t* member_dev, int32_t* num_steps_dev, int64_t n_envs, float* next_state_dev,
                      float* disc_dev, uint8_t* done_dev, const float* w_dev, float lambda_b, float threshold,
                      float c_min, float c_max, int32_t clamp_cost, float* cost_dev, float* ipm_dev,
                      float* bonus_dev, void* stream);

/* ---- MILO cost on explicit rows ---------------------------------------- */

/* RBFLinearCost.get_rep (LC:64-71): phi_dev [E][D] = cos(x W^T + b)*sqrt(2/D),
 * x_dev [E][in_dim].  phi_sum_dev [D] (may be NULL) receives sum_e phi, the
 * numerator of fit_cost's mean (LC:88). */
int simstep_rff_features(simstep_handle* h, const float* x_dev, int64_t n_rows, float* phi_dev,
                         double* phi_sum_dev, void* stream);

/* RBFLinearCost.get_costs (LC:96-103) before the clamp: dot_dev[e] = phi(x_e).w */
int simstep_rff_dot(simstep_handle* h, const float* x_dev, int64_t n_rows, const float* w_dev, float* dot_dev,
                    void* stream);

/* RBFLinearCost.get_bonus_costs (LC:111-152) given rows and their discrepancy. */
int simstep_bonus_cost(simstep_handle* h, const float* x_dev, const float* disc_dev, int64_t n_rows,
                       const float* w_dev, float lambda_b, float threshold, float c_min, float c_max,
                       int32_t clamp_cost, float* cost_dev, float* ipm_dev, float* bonus_dev, void* stream);

/* ---- DeepMimic imitation reward ----------------------------------------- */

/* Articulated character of the reward (humanoid3d.txt Skeleton/BodyDefs):
 * joints are topologically ordered, joint 0 is the root. */
typedef struct simstep_character {
  int32_t n_joints;
  int32_t joint_type[SIMSTEP_MAX_JOINTS];   /* 0 root(none) 1 spherical 2 revolute 3 fixed */
  int32_t parent[SIMSTEP_MAX_JOINTS];
  float attach[SIMSTEP_MAX_JOINTS][3];      /* joint AttachX/Y/Z                */
  int32_t param_offset[SIMSTEP_MAX_JOINTS]; /* offset in pose/vel (KT:1053-1062) */
  int32_t is_end_eff[SIMSTEP_MAX_JOINTS];
  float diff_weight[SIMSTEP_MAX_JOINTS];    /* DiffWeight (SI:300-312 normalises) */
  float body_mass[SIMSTEP_MAX_JOINTS];
  float body_attach[SIMSTEP_MAX_JOINTS][3]; /* BodyDefs AttachX/Y/Z             */
  int32_t dof;                              /* pose/vel length, 43              */
} simstep_character;

/* Reference clip after cMotion::Load post-processing (Motion.cpp:356-442) and
 * the first-frame centring of KinController.cpp:144-160: frames_host
 * [n_frames][dof] poses, frame_vel_host [n_frames][dof] (Motion.cpp:170-191),
 * frame_time_host [n_frames] start times, loop_wrap != 0 for "Loop":"wrap",
 * cycle_delta = root translation of one cycle (KinController.cpp:162-175). */
int simstep_load_clip(simstep_handle* h, const simstep_character* ch, int32_t n_frames,
                      const float* frames_host, const float* frame_vel_host, const float* frame_time_host,
                      float duration, int32_t loop_wrap, const float* cycle_delta_host);

/* Batched cSceneImitate::CalcRewardImitate (SI:7-127) against the loaded clip.
 *   pose_dev, vel_dev [E][dof]   simulated character (KT pose/vel layout)
 *   kin_time_dev [E]             clip time of env e's kinematic character
 *   kin_origin_dev [E][3] or NULL world offset of the kin character's origin
 *   reward_dev [E]; terms_dev [E][5] (pose, vel, end_eff, root, com rewards) or NULL */
int simstep_imitation_reward(simstep_handle* h, const float* pose_dev, const float* vel_dev,
                             const float* kin_time_dev, const float* kin_origin_dev, int64_t n_envs,
                             float* reward_dev, float* terms_dev, void* stream);

/* cKinCharacter pose/vel at a clip time (KinCharacter.cpp:573-640 via
 * Motion.cpp:267-305): out_pose_dev, out_vel_dev [E][dof]. */
int simstep_clip_sample(simstep_handle* h, const float* kin_time_dev, const float* kin_origin_dev, int64_t n_envs,
                        float* out_pose_dev, float* out_vel_dev, void* stream);

/* Character state features of the env (DeepMimicCore sim/CtController.cpp:378-495, BuildStatePose /
 * BuildStateVel: what SimEnv.reset() reads through record_state, sim_env.py:270-285) from generalized
 * pose_dev / vel_dev [n][dof] of the character loaded with simstep_load_clip, body transforms taken
 * kinematically from the pose (the simulator's state right after SetPose / SetVel), ground plane y = 0:
 * state_dev [n][1 + 15 * n_joints] = root height | per body (pos[3], normal[3], tangent[3]) | per body
 * (lin vel[3], ang vel[3]).  The Record* arguments mirror the controller file's RecordAllWorld /
 * RecordWorldRootPos / RecordWorldRootRot; vel_scale = 1, or 1 / UpdateRate for RecordVelAsPos. */
int simstep_record_state(simstep_handle* h, const float* pose_dev, const float* vel_dev, int64_t n_envs,
                         int32_t record_all_world, int32_t record_world_root_pos, int32_t record_world_root_rot,
                         float vel_scale, float* state_dev, void* stream);

/* MLPCost's feature map (milo/milo/linear_cost.py:154-222): a plain MLP
 *   x -> act(W_0 x + b_0) -> ... -> act(W_{L-1} . + b_{L-1}) -> tanh(W_head . + b_head) -> cos(.) * sqrt(2/D)
 * on a handle created with state_dim = input width, action_dim = 0, n_models = 1, hidden = the MLP's
 * hidden sizes, dense_connect = 0, transform = 0.  weights_host[l] / biases_host[l], l < n_hidden, are the
 * hidden nn.Linear layers; head_weight_host [feature_dim][hidden[L-1]] / head_bias_host the last nn.Linear;
 * head_mode selects what follows it (SIMSTEP_HEAD_*, below): tanh then the cosine features as in the
 * reference's MLPCost (linear_cost.py:208-236), or nothing (a discriminator's raw output).  Afterwards
 * simstep_rff_features / simstep_rff_dot / simstep_bonus_cost evaluate this feature map (x_dev rows are
 * state_dim wide); simstep_step* are not available on such a handle. */
int simstep_load_feature_net(simstep_handle* h, const float* const* weights_host, const float* const* biases_host,
                             int32_t feature_dim, const float* head_weight_host, const float* head_bias_host,
                             int32_t head_mode);

/* head_mode of simstep_load_feature_net */
#define SIMSTEP_HEAD_TANH_COS 1 /* MLPCost: cos(tanh(.)) * sqrt(2/D) */
#define SIMSTEP_HEAD_LINEAR 2   /* the last nn.Linear's output itself: GAIL discriminator, gail_cost.py:18-43 */

/* What simstep_rff_dot / simstep_bonus_cost do with the per-row value d = phi(x) . w before the bonus
 * combine (default SIMSTEP_COST_IDENTITY).  With a LINEAR head of width 1 and w = [1], d is the
 * discriminator output and the two GAIL settings give GAILCost.get_ls_costs / get_ll_costs
 * (milo/milo/gail_cost.py:232-246); simstep_bonus_cost with clamp_cost = 0 then is
 * GAILCost.get_bonus_costs (gail_cost.py:255-283): cost = (1 - lambda_b) c(d) - lambda_b * disc. */
#define SIMSTEP_COST_IDENTITY 0
#define SIMSTEP_COST_GAIL_LS 1 /* -(max(1 - 0.25 (1 - d)^2, 0)) */
#define SIMSTEP_COST_GAIL_LL 2 /* logsigmoid(d) */
int simstep_set_cost_transform(simstep_handle* h, int32_t transform);

/* ---- on-device rollout helpers ------------------------------------------ */

/* Gaussian MLP policy of mjrl (mjrl/mjrl/policies/gaussian_mlp.py:6-104 over
 * mjrl/mjrl/utils/fc_network.py:9-55): n_layers linear layers, weights_host[l] is
 * fc_layers.l.weight [layer_out[l]][layer_in[l]] row-major, biases_host[l] its bias;
 * tanh_act selects tanh (1) or relu (0) between layers; in_shift/in_scale [obs],
 * out_shift/out_scale [act] are FCNetwork's transformations (NULL: 0 / 1);
 * log_std_host [act] is the policy's log standard deviation (NULL: deterministic). */
int simstep_load_policy(simstep_handle* h, int32_t n_layers, const int32_t* layer_in, const int32_t* layer_out,
                        const float* const* weights_host, const float* const* biases_host, int32_t tanh_act,
                        const float* in_shift_host, const float* in_scale_host, const float* out_shift_host,
                        const float* out_scale_host, const float* log_std_host);

/* Batched MLP.get_action (gaussian_mlp.py:95-104): mean_dev [E][act] = model(obs),
 * action_dev [E][act] = mean + exp(log_std) * noise_dev[e] (noise_dev: standard normal
 * draws supplied by the caller, NULL: action = mean, the 'evaluation' action).
 * Either output may be NULL. */
int simstep_policy_act(simstep_handle* h, const float* obs_dev, const float* noise_dev, int64_t n_envs,
                       float* action_dev, float* mean_dev, void* stream);

/* Discounted sums over time-major [T][E] arrays (mjrl/mjrl/utils/process_samples.py:3-45):
 * returns = discount_sum(reward, gamma); advantages = GAE(gamma, gae_lambda) against
 * baseline_dev [T][E].  An env's column holds one or more trajectories back to back:
 * seg_end_dev [T][E] (NULL: none) != 0 marks the last step of a trajectory that terminated
 * (milo/milo/sampler.py:79 stores terminated=done); the trailing trajectory ends at
 * len_dev[e]-1 (NULL: T) and bootstraps from its last baseline value unless
 * terminated_dev[e] != 0 (NULL: not terminated).  Entries at t >= len are written as 0.
 * returns_dev / advantages_dev may be NULL. */
int simstep_discount(simstep_handle* h, const float* reward_dev, const float* baseline_dev, const uint8_t* seg_end_dev,
                     const int32_t* len_dev, const uint8_t* terminated_dev, int32_t T, int64_t n_envs, float gamma,
                     float gae_lambda, float* returns_dev, float* advantages_dev, void* stream);

/* Between two steps of a rollout (milo/milo/sampler.py:36-66 calls env.reset() when a
 * trajectory ends; gym-simenv/gym_simenv/envs/sim_env.py:270-285): for every env
 *   done_dev[e] ? state_out[e] = pool_dev[pick_dev[e] mod n_pool], num_steps[e] = 0,
 *                 member[e] = (member[e] + 1) mod n_models
 *               : state_out[e] = next_state[e].
 * pool_dev [n_pool][state_dim] holds caller-supplied initial states (the reference draws
 * them from the DeepMimic simulator, which stays outside this library). */
int simstep_auto_reset(simstep_handle* h, const float* next_state_dev, const uint8_t* done_dev, const float* pool_dev,
                       const int32_t* pick_dev, int32_t n_pool, int64_t n_envs, float* state_out_dev,
                       int32_t* member_dev, int32_t* num_steps_dev, void* stream);

/* Advantage whitening (mjrl/mjrl/utils/process_samples.py:14-19, 31-36) in two calls so that a
 * multi-GPU caller can all-reduce between them:
 *   simstep_moments: out_dev[0..2] = {count, sum, sum of squares} (fp64) of x_dev[i] over the entries
 *                    with valid_dev[i] != 0 (NULL: all n entries); deterministic two-pass reduction.
 *   simstep_whiten:  out_dev[i] = (x[i] - mean) / (std + eps), mean = sum/count, std = population
 *                    standard deviation (numpy's .std()), from stats_dev = {count, sum, sumsq};
 *                    masked-out entries are written as 0.  out_dev may alias x_dev. */
int simstep_moments(simstep_handle* h, const float* x_dev, const uint8_t* valid_dev, int64_t n, double* out_dev,
                    void* stream);
int simstep_whiten(simstep_handle* h, const float* x_dev, const uint8_t* valid_dev, int64_t n, const double* stats_dev,
                   float eps, float* out_dev, void* stream);

/* ---- natural policy gradient step of the loaded policy (mjrl/mjrl/algos/npg_cg.py: NPG.train_from_paths) ---- */

/* One NPG update of the policy loaded with simstep_load_policy, computed from rows of (obs, action, advantage) in
 * device memory, written in place into the handle's policy (nothing is re-allocated: graphs that captured
 * simstep_policy_act stay valid).  The calls only enqueue work; the "sums" they return are un-normalised, with their
 * row counts, so that a multi-GPU caller can all-reduce them between calls.  P is the length of the parameter vector
 * in mjrl's get_param_values order: per linear layer the weight [out][in] then the bias [out], then log_std [act].
 *   init:    allocates the NPG state for the loaded policy (*n_params_out = P); EINVAL when the parameter vector does
 *            not fit the per-CTA gradient accumulator.  min_log_std is MLP.min_log_std (the clamp of set_param_values).
 *            simstep_load_policy discards this state.
 *   params:  set != 0: theta_dev [P] fp32 becomes the parameters (and is written into the policy); set == 0: copies
 *            the current parameters to theta_dev.
 *   grad:    out_dev [P + 2] fp64 = { sum_i adv_i dLL_i/dtheta, rows, sum_i adv_i } over the rows with valid_dev[i] != 0
 *            (NULL: all n rows); LL is MLP.log_likelihood.
 *   prepare: caches the hidden activations of the Fisher rows: obs rows idx_dev[0 .. n_idx) (int64), or all n rows when
 *            idx_dev is NULL.  Call again whenever the rows or the parameters change.
 *   fvp:     out_dev [P + 2] fp64 = { sum over Fisher rows of H_i v, rows, 0 }, H_i the Hessian of MLP.mean_kl at new =
 *            old for row i (rows with valid_dev[idx] == 0 do not count); v_dev [P] fp64, or NULL for the direction
 *            of the CG solve, in which case nothing is computed once the solve has converged.
 *   cg:      SIMSTEP_NPG_CG_START with the grad sums: g = sum / rows, x = 0, r = p = g (cg_solve.py);
 *            SIMSTEP_NPG_CG_STEP with the fvp sums of the direction: one cg_solve iteration with
 *            F p = sum / rows + damping * p; converged (remaining steps are no-ops) once r.r < 1e-10.
 *   apply:   theta += alpha * x with alpha = const_lr ? step : sqrt(|step / (g.x + 1e-10)|), log_std clamped at
 *            min_log_std, written into the policy; the previous parameters are kept for diag.
 *   diag:    out_dev [3] fp64 = { rows, sum_i exp(LL_new - LL_old) adv_i, sum_i KL_i(new, old) } (CPI_surrogate and
 *            kl_old_new of the step just applied).
 *   scalars: out_dev [6] fp64 = { r.r, g.x, alpha, gradient rows, mean advantage, CG iterations run }. */
#define SIMSTEP_NPG_CG_START 0
#define SIMSTEP_NPG_CG_STEP 1
int simstep_npg_init(simstep_handle* h, float min_log_std, int64_t* n_params_out);
int simstep_npg_params(simstep_handle* h, int32_t set, float* theta_dev, void* stream);
int simstep_npg_grad(simstep_handle* h, const float* obs_dev, const float* act_dev, const float* adv_dev,
                     const uint8_t* valid_dev, int64_t n, double* out_dev, void* stream);
int simstep_npg_prepare(simstep_handle* h, const float* obs_dev, int64_t n, const int64_t* idx_dev, int64_t n_idx,
                        void* stream);
int simstep_npg_fvp(simstep_handle* h, const float* obs_dev, const uint8_t* valid_dev, int64_t n, const int64_t* idx_dev,
                    int64_t n_idx, const double* v_dev, double* out_dev, void* stream);
int simstep_npg_cg(simstep_handle* h, int32_t op, const double* sums_dev, double damping, void* stream);
int simstep_npg_apply(simstep_handle* h, double step, int32_t const_lr, void* stream);
int simstep_npg_diag(simstep_handle* h, const float* obs_dev, const float* act_dev, const float* adv_dev,
                     const uint8_t* valid_dev, int64_t n, double* out_dev, void* stream);
int simstep_npg_scalars(simstep_handle* h, double* out_dev, void* stream);

/* ---- ensemble training (milo/milo/dynamics.py:236-250, DynamicsModel.train_step) ------------------- */

/* All n_models members take one optimisation step per call, each on its own batch of batch_rows
 * transitions: forward on normalised inputs (unnormalize_out = False), MSE against the normalised state
 * difference, backward, optional gradient-norm clipping at grad_clip per member, then one of the reference's
 * optimisers (dynamics.py:198-203): SGD with Nesterov momentum (optimizer = 0; lr, momentum) or Adam
 * (optimizer = 1; lr, momentum = beta1, beta2, eps), with the update rules of the optimiser library it uses.
 * The handle must have been created with SIMSTEP_PREC_TF32: the fp32 parameters inside the handle are
 * the master copy and the tensor-core operands at once.  Call simstep_train_init BEFORE
 * simstep_load_ensemble so that the parameters are stored with all their bits.
 *   state_dev / next_state_dev [n_models][batch_rows][state_dim], action_dev [n_models][batch_rows][action_dim]
 *   loss_dev [n_models] fp64: each member's mean-squared error on its batch (before the update)
 * simstep_train_loss is DynamicsModel.validate_step (dynamics.py:252-262): forward + loss only.
 * simstep_train_grads runs forward + backward and leaves the gradients in the handle (no update).
 * simstep_train_export copies parameters, the last gradients or the first optimiser moment (SGD momentum
 * buffer / Adam exp_avg) back in nn.Linear layout: weights_host[m * n_layers + l] -> float[out][in],
 * biases_host[...] -> float[out] (NULL entries are skipped). */
#define SIMSTEP_TRAIN_PARAMS 0
#define SIMSTEP_TRAIN_GRADS 1
#define SIMSTEP_TRAIN_MOMENTS 2
int simstep_train_init(simstep_handle* h, int32_t max_batch_rows, int32_t optimizer, float lr, float momentum,
                       float beta2, float eps);
int simstep_train_step(simstep_handle* h, const float* state_dev, const float* action_dev, const float* next_state_dev,
                       int32_t batch_rows, float grad_clip, double* loss_dev, void* stream);
int simstep_train_loss(simstep_handle* h, const float* state_dev, const float* action_dev, const float* next_state_dev,
                       int32_t batch_rows, double* loss_dev, void* stream);
int simstep_train_grads(simstep_handle* h, const float* state_dev, const float* action_dev, const float* next_state_dev,
                        int32_t batch_rows, double* loss_dev, void* stream);
int simstep_train_export(simstep_handle* h, int32_t what, float* const* weights_host, float* const* biases_host);

/* ---- reductions used by the multi-GPU host code ------------------------- */

/* counts_dev[b] (int64, bins entries, overwritten) = number of x_dev[i] in [lo, hi] whose bin
 * clamp(floor((x - lo) / ((hi - lo) / bins)), 0, bins - 1) is b; 1 <= bins <= 8192.  The all-reduced
 * histograms of the ranks give the global discrepancy quantile without gathering samples. */
int simstep_histogram(simstep_handle* h, const float* x_dev, int64_t n, double lo, double hi, int32_t bins,
                      int64_t* counts_dev, void* stream);

/* Device-side steps of the distributed q-quantile (amp_extensions_b200.parallel.global_quantile): the windows that
 * bracket the two order statistics live in device memory, so a refinement costs no host round trip.
 * qstate_dev: 8 doubles, for order statistic i in {0, 1}: [4i] window lo, [4i+1] window hi, [4i+2] number of
 * samples below the window, [4i+3] rank k of the order statistic.  Every op only enqueues work on `stream`.
 *   MINMAX: out_dev[0] = -min(x), out_dev[1] = max(x)              (one all-reduce MAX makes both global)
 *   HIST:   counts_dev[i*bins + b] (int64, overwritten) = samples of window i in bin b, 1 <= bins <= 4096
 *   SELECT: narrows both windows to the bin that holds their order statistic, given the (all-reduced) counts
 *   WINMIN: out_dev[i] = -min{x in window i}                       (all-reduce MAX, negate: the order statistic) */
#define SIMSTEP_QOP_MINMAX 0
#define SIMSTEP_QOP_HIST 1
#define SIMSTEP_QOP_SELECT 2
#define SIMSTEP_QOP_WINMIN 3
int simstep_quantile_op(simstep_handle* h, int32_t op, const float* x_dev, int64_t n, int32_t bins, double* qstate_dev,
                        int64_t* counts_dev, double* out_dev, void* stream);

/* out_dev[0] = max_e x[e], out_dev[1] = sum_e x[e] (fp64 accumulate), n may be 0. */
int simstep_reduce_max_sum(simstep_handle* h, const float* x_dev, int64_t n, double* out_dev, void* stream);

/* ---- measurement ---------------------------------------------------------- */

/* Device time per kernel category, measured with CUDA events recorded on the
 * launch stream around each launch (bench.py's roofline numbers).  Recording is
 * off by default; enable, run, then read (read synchronises the device). */
#define SIMSTEP_PROF_PREP 0          /* input normalisation / operand pack      */
#define SIMSTEP_PROF_ENSEMBLE_GEMM 1 /* all layer GEMMs of one ensemble pass    */
#define SIMSTEP_PROF_POST 2          /* next state + discrepancy + termination  */
#define SIMSTEP_PROF_RFF_PACK 3
#define SIMSTEP_PROF_RFF_GEMM 4
#define SIMSTEP_PROF_COMBINE 5
#define SIMSTEP_PROF_IMITATION 6
#define SIMSTEP_PROF_CATEGORIES 8
int simstep_profile_enable(simstep_handle* h, int32_t enable);
/* ms_out[SIMSTEP_PROF_CATEGORIES] accumulated milliseconds, count_out[...] number
 * of bracketed regions; reset != 0 clears the accumulators afterwards. */
int simstep_profile_read(simstep_handle* h, double* ms_out, int64_t* count_out, int32_t reset);

/* ---- debugging / unit tests -------------------------------------------- */

/* One grouped GEMM through the production tcgen05 kernel:
 * d[g][m][n] = sum_k a[g][m][k]*b[g][n][k] (+bias[g][n]) for g < groups,
 * a_dev [groups][m][k], b_dev [groups][n][k], d_dev [groups][m][n] fp32.
 * Operands are rounded to `precision` exactly as the ensemble path does. */
int simstep_debug_gemm(int32_t precision, int32_t groups, int64_t m, int32_t n, int32_t k, const float* a_dev,
                       const float* b_dev, const float* bias_dev, float* d_dev, void* stream);

/* Number of kernels this library has launched on the calling process. */
int64_t simstep_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SIMSTEP_H_ */
