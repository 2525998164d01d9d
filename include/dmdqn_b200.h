/*
 * dmdqn_b200.h -- C ABI of the B200-native agent-side hot path of dmdqn.
 *
 * The reference (pranshu-raj-211/dmdqn) is pure Python on TensorFlow/Keras and has NO
 * FFI / plugin interface; this header is the new, thin seam (SURVEY.md section 8, row B2).
 * Every entry point names the reference function(s) whose arithmetic it replaces; the
 * Python side (dmdqn_b200/agent.py, group.py) keeps the reference's class and method
 * names on top of these calls.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer owned by
 *     the caller (the Python host allocates them as torch tensors); the library keeps no
 *     state and allocates nothing.
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no host sync),
 *     so they can be captured into a CUDA graph.
 *   - return value: DMDQN_OK or a negative error code; dmdqn_last_error() gives the
 *     thread-local message.  Nothing aborts, nothing throws (the reference never raises
 *     on this path either: it returns None/0 or drops the sample -- dqn_agent.py:50-54,
 *     61-62,333-335).
 *   - there is no CPU fallback: without a CUDA device every compute call fails with
 *     DMDQN_ERR_CUDA.
 *
 * Device data layout (see DESIGN.md "Data layout in HBM")
 *   replay ring, per agent a (deque(maxlen=C), dqn_agent.py:27-57):
 *     obs, next_obs : float [n_agents][capacity][obs_stride]   (obs_stride = obs_dim rounded
 *                      up to 16 floats: 89 -> 96 = three 128-byte lines; pad columns are 0)
 *     act           : int32 [n_agents][capacity]
 *     rew           : double[n_agents][capacity]   (the reference keeps Python floats)
 *     done          : uint8 [n_agents][capacity]
 *     n_written     : int64 [n_agents]             (slot of next write = n_written % capacity)
 *   network parameters, per network g (Keras kernel layout [in,out], y = xW + b,
 *   dqn_agent.py:153-184), one contiguous block of dmdqn_layout.stride floats:
 *     W1[obs_stride][H] | b1[H] | W2[H][H] | b2[H] | W3[H][4] | b3[4] | pad
 *   theta, theta_tgt, adam_m, adam_v all use that block layout; learn_step: int32[n_nets].
 *   dueling networks (dmdqn_hparams.dueling = 1; dmdqn_param_layout_dueling) append the value head after b3:
 *     W1 | b1 | W2 | b2 | W3[H][4] | b3[4] | wv[H] | bv | pad[3] | pad
 *   with the same offsets up to b3, wv at b3 + 4 (16-byte aligned), bv at b3 + 4 + H, Adam over [0, b3 + 8 + H) (the
 *   three pad floats keep gradient 0 and stay 0) and the stride rounded up to 32 floats.  Q is
 *     Q(s, a) = V(s) + Adv(s, a) - (1/A) sum_{b<A} Adv(s, b),  Adv = h2 . W3[:, a] + b3[a],  V = h2 . wv + bv
 *   (Wang et al. 2016), which is the plain 4-wide head with the effective weights
 *     W3e[k][a] = (W3[k][a] - mean_{b<A} W3[k][b]) + wv[k]  (a < A; 0 for a >= A),  b3e[a] = (b3[a] - mean_{b<A} b3[b]) + bv
 *   each mean summed left to right in fp32 and divided by A (IEEE division).  Advantage columns >= A keep gradient 0.
 */
#ifndef DMDQN_B200_H
#define DMDQN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMDQN_ABI_VERSION 3

#define DMDQN_OK            0
#define DMDQN_ERR_ARG      -1   /* bad dims / null pointer / unsupported size          */
#define DMDQN_ERR_CUDA     -2   /* CUDA runtime error (no device, launch failure, ...) */
#define DMDQN_ERR_WORKSPACE -3  /* workspace too small                                  */

#define DMDQN_LOSS_MSE   0      /* dqn_agent.py:141,352 (reference default)  */
#define DMDQN_LOSS_HUBER 1      /* experimental/agent.py:99, delta = 1       */

#define DMDQN_SAMPLE_INDICES     0  /* host supplies logical indices (e.g. CPython random.sample) */
#define DMDQN_SAMPLE_FISHER_YATES 1 /* uint32 draws, without replacement (partial Fisher-Yates)   */
#define DMDQN_SAMPLE_REPLACEMENT 2  /* uint32 draws, with replacement (deviation, flagged)        */
#define DMDQN_SAMPLE_PRIORITIZED 3  /* uint32 draws, proportional prioritized replay (see below)   */

#define DMDQN_ADAM_KERAS 0      /* eps = adam_eps                       (keras 3.9.2)      */
#define DMDQN_ADAM_TORCH 1      /* eps = adam_eps * sqrt(1 - beta2^t)   (torch.optim.Adam) */

#define DMDQN_PRECISION_FP32   0 /* FFMA, fp32 accumulate                                                   */
#define DMDQN_PRECISION_TF32   1 /* tcgen05 kind::tf32, one MMA per product (~1e-3; toleranced separately)   */
#define DMDQN_PRECISION_TF32X3 2 /* tcgen05 kind::tf32, error-compensated hi/lo split, 3 MMAs per product:   */
                                 /* fp32-class accuracy on the tensor cores (H = 256 only)                   */

#define DMDQN_MAX_ACTIONS 4
#define DMDQN_OWN_DIM 17        /* order_lanes.py:430-499 */
#define DMDQN_OBS_DIM 89        /* order_lanes.py:502-555 */
#define DMDQN_PHASE_LUT 16

typedef struct dmdqn_dims {
    int32_t n_agents;    /* replay rings (intersections) held by this GPU                   */
    int32_t n_nets;      /* independent networks: n_agents, or 1 when parameters are shared */
    int32_t obs_dim;     /* D  (89)                                                         */
    int32_t obs_stride;  /* floats per stored observation row; multiple of 16, >= obs_dim   */
    int32_t hidden;      /* H in {64,128,256,512}; nn_layers = [H, H]                       */
    int32_t n_actions;   /* A <= 4                                                          */
    int32_t batch;       /* B, transitions per network per learn step                       */
    int32_t capacity;    /* C, ring capacity per agent                                      */
} dmdqn_dims;

typedef struct dmdqn_layout {   /* float offsets inside one parameter block */
    int64_t w1, b1, w2, b2, w3, b3, stride;
} dmdqn_layout;

typedef struct dmdqn_replay {   /* all device pointers */
    float*   obs;
    float*   next_obs;
    int32_t* act;
    double*  rew;
    uint8_t* done;
    int64_t* n_written;
    /* Prioritized replay (DMDQN_SAMPLE_PRIORITIZED; NULL = none, every other mode ignores them):
     *   priority     float[n_agents][capacity]  p^alpha of each PHYSICAL slot; 0 = never written (never drawn)
     *   priority_max float[n_agents]            largest priority seen by the agent's ring; the host starts it at 1.0
     * dmdqn_push writes priority_max[a] into the slot it fills; the learn step writes the new priority of every
     * sampled row (see dmdqn_learn). */
    float*   priority;
    float*   priority_max;
} dmdqn_replay;

typedef struct dmdqn_nets {     /* all device pointers */
    float*   theta;
    float*   theta_tgt;
    float*   adam_m;
    float*   adam_v;
    int32_t* learn_step;
} dmdqn_nets;

typedef struct dmdqn_hparams {
    double  gamma;                    /* agent_config.yaml: gamma (rounded to fp32 on use) */
    double  learning_rate;            /* agent_config.yaml: learning_rate                  */
    double  beta1, beta2, adam_eps;   /* Keras Adam defaults 0.9, 0.999, 1e-7; the step    */
                                      /* size alpha_t is evaluated in float64 on the device */
    double  tau;                      /* < 0: hard sync every target_update_frequency      */
                                      /* >= 0: Polyak every step (dqn_agent.py:389-399)    */
    int32_t target_update_frequency;  /* agent_config.yaml: target_update_frequency        */
    int32_t loss;                     /* DMDQN_LOSS_*                                      */
    int32_t normalize_rewards;        /* 1 = per-batch z-score (dqn_agent.py:66-69)        */
    int32_t double_dqn;               /* 1 = dqn_agent.py:342-345, 0 = experimental/agent.py:166-167 */
    int32_t adam_form;                /* DMDQN_ADAM_*                                      */
    int32_t sample_mode;              /* DMDQN_SAMPLE_*                                    */
    int32_t precision;                /* DMDQN_PRECISION_*                                 */
    int32_t dueling;                  /* 0 = plain head, 1 = dueling value + advantage heads (parameter blocks in the
                                         dueling layout); any other value is refused.  In what was interior padding:
                                         offset 76, sizeof stays 112 */
    /* prioritized replay (read in DMDQN_SAMPLE_PRIORITIZED only): priority = (|delta| + per_eps)^per_alpha,
     * importance exponent beta_t = min(1, per_beta0 + (1 - per_beta0) * t / per_beta_steps) with t the network's
     * learn_step after the increment (per_beta_steps <= 0: beta_t = per_beta0) */
    double  per_alpha, per_beta0, per_eps;
    int32_t per_beta_steps;
    /* n-step returns (every sample mode; see dmdqn_sample): transitions per TD target, 0 or 1 = one-step,
     * at most DMDQN_MAX_NSTEP.  Placed in what was the struct's tail padding: offset 108, sizeof stays 112. */
    int32_t n_step;
} dmdqn_hparams;
#define DMDQN_MAX_NSTEP 16

/* Per-network learn outputs, 8 floats each: loss, q_mean, q_std (population, over the
 * [B,A] online Q of the sampled states), action histogram[4], learned flag (0/1)
 * (dqn_agent.py:359-370). */
#define DMDQN_METRICS_STRIDE 8

const char* dmdqn_last_error(void);
int dmdqn_abi_version(void);

/* Parameter block layout for the given dims. */
int dmdqn_param_layout(const dmdqn_dims* dims, dmdqn_layout* out);

/* Parameter block layout of a dueling network (dmdqn_hparams.dueling = 1): dmdqn_param_layout's offsets up to b3, the
 * value head's wv[H] and bv, and the dueling stride.  Every call that takes dueling blocks and no hparams has a
 * *_dueling sibling below; passing dueling blocks to dmdqn_act or dmdqn_sync_target is a caller error. */
typedef struct dmdqn_dueling_layout {
    int64_t w1, b1, w2, b2, w3, b3, wv, bv, stride;
} dmdqn_dueling_layout;
int dmdqn_param_layout_dueling(const dmdqn_dims* dims, dmdqn_dueling_layout* out);

/* Bytes of device scratch dmdqn_sample / dmdqn_learn need for these dims. */
int dmdqn_workspace_bytes(const dmdqn_dims* dims, size_t* out_bytes);

/* K0 -- observation + reward featurisation for all intersections.
 * Replaces get_own_state / _get_neighbor_info / build_state_vector
 * (src/experimental/order_lanes.py:392-555) and calculate_local_reward /
 * calculate_global_reward + the 0.3/0.7 mix (src/scripts/train.py:159-165,241,251-254).
 *   halting      device int32 [n][12]   slot = dir*3+lane (n,s,e,w); -1 = lane absent
 *   phase        device int32 [n]       SUMO phase index
 *   next_switch  device double[n], phase_dur device double[n], sim_time: TraCI readings
 *   signal_valid device uint8 [n]       0 -> phase/time stay [0,0,0,0,-1] (shipped behaviour)
 *   nbr_idx      device int32 [n][4]    neighbour rows in n,s,e,w order, -1 = none
 *   phase_lut    device int32 [16]      phase index -> one-hot slot 0..3 or -1
 *   snapshot     device double[n][17] or NULL: neighbour blocks come from this
 *                global_state snapshot (order_lanes.py:547-548) instead of the live blocks
 *   own_out      device double[n][17]   (the caller's next global_state)
 *   obs_out      device float [n][obs_out_stride]  first 89 columns written, rest zeroed
 *   reward_out   device double[n], global_out device double[1]: reward from THESE readings
 *                used as the pre-step state (train.py:241).
 *   scratch      device int64 [2], zero on entry; left zero on return. */
int dmdqn_featurize(int32_t n, const int32_t* halting, const int32_t* phase,
                    const double* next_switch, const double* phase_dur, double sim_time,
                    const uint8_t* signal_valid, const int32_t* nbr_idx, const int32_t* phase_lut,
                    const double* snapshot, double local_weight, double global_weight,
                    double* own_out, float* obs_out, int32_t obs_out_stride,
                    double* reward_out, double* global_out, int64_t* scratch, void* stream);

/* K0, second layout -- replaces SumoTrafficEnvironment._get_local_observation / _get_observations /
 * _get_neighbor_presence_vector / _calculate_rewards (reference src/agents/sumo_env.py:532-580,582-631,633-645,
 * 652-679): the 74-dim observation local(14) | presence(4: N,E,S,W) | 4 x neighbour local(14), pad -1.0, and the
 * queue-reduction reward.
 *   halting      device int32 [n][12]   queues in N,E,S,W order x 3 lanes; -2 = PAD lane (-> 0.0), -1 = failed read (-> -1.0)
 *   phase        device int32 [n], next_switch device double[n], sim_time
 *   signal_valid device uint8 [n]       0 -> both signal slots keep the -1.0 padding value
 *   nbr_idx      device int32 [n][4]    neighbour rows in N,E,S,W order, -1 = none / not controlled
 *   prev_own     device double[n][14] or NULL (first step): the previous call's own_out
 *   own_out      device double[n][14] or NULL
 *   obs_out      device float [n][obs_out_stride]  first 74 columns written, rest zeroed
 *   reward_out   device double[n] or NULL: sum max(0, prev queues) - sum max(0, current queues); 0 when prev_own is NULL */
#define DMDQN_OWN_ALT_DIM 14
#define DMDQN_OBS_ALT_DIM 74
int dmdqn_featurize_alt(int32_t n, const int32_t* halting, const int32_t* phase, const double* next_switch,
                        const uint8_t* signal_valid, double sim_time, const int32_t* nbr_idx, const double* prev_own,
                        double* own_out, float* obs_out, int32_t obs_out_stride, double* reward_out, void* stream);

/* K2 -- batched epsilon-greedy action selection, one observation per agent.
 * Replaces DQNAgent.select_action (src/agents/dqn_agent.py:263-274; the epsilon schedule
 * :258-261 stays on the host) and select_greedy_action (experimental/agent.py:148-152).
 *   obs        device float [n_agents][obs_in_stride]
 *   eps        device double[n_agents]   host-computed epsilon per agent
 *   w_explore, w_action  device uint32[n_agents]  supplied draws: explore iff
 *              w_explore < eps * 2^32; random action = (w_action * A) >> 32
 *   actions_out device int32[n_agents];  q_out device float[n_agents][4] or NULL
 *              (q_out rows of exploring agents are left untouched: the reference skips
 *              the forward pass when exploring). */
int dmdqn_act(const dmdqn_dims* dims, const dmdqn_nets* nets, const float* obs, int32_t obs_in_stride,
              const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
              int32_t* actions_out, float* q_out, void* stream);
/* The same on dueling parameter blocks: the head is folded into W3e / b3e in registers with the arithmetic above, so
 * q_out and the actions equal dmdqn_act's on a plain block holding the folded head, bit for bit. */
int dmdqn_act_dueling(const dmdqn_dims* dims, const dmdqn_nets* nets, const float* obs, int32_t obs_in_stride,
                      const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
                      int32_t* actions_out, float* q_out, void* stream);

/* K1a -- append one transition per agent to its ring.
 * Replaces ReplayBuffer.add / DQNAgent.remember / store_experience
 * (src/agents/dqn_agent.py:31-57,306-325).  mask (device uint8[n_agents] or NULL)
 * selects the agents that store. */
int dmdqn_push(const dmdqn_dims* dims, const dmdqn_replay* replay, const float* obs,
               const int32_t* act, const double* rew, const float* next_obs, const uint8_t* done,
               int32_t in_stride, const uint8_t* mask, void* stream);

/* K1b -- draw the batch of every network and z-score its rewards.
 * Replaces ReplayBuffer.sample (src/agents/dqn_agent.py:59-85) up to the gather.
 *   draws  device [n_nets][batch]: int32 logical indices (0 = oldest) or uint32 words,
 *          per hp->sample_mode
 *   learn_mask device uint8[n_nets] or NULL; a network is "active" iff its mask is set
 *          and its ring(s) hold >= batch transitions (dqn_agent.py:61-62,333-335).
 *   advance_step: 1 when called as the first stage of a learn step (bumps learn_step of
 *          active networks, dqn_agent.py:359); 0 for a stand-alone sample().
 * Results stay in the workspace (rows, r_hat, actions, dones, active flags).
 *
 * DMDQN_SAMPLE_PRIORITIZED (proportional prioritized replay, Schaul et al. 2016; independent networks only, and
 * replay->priority must be set; capacity <= DMDQN_PER_MAX_CAPACITY).  Network g draws from agent g's ring:
 *   1. S = sum of priority[g][0..C) in float64: chunks of 128 consecutive slots, each summed as lane l (0..31) adding
 *      slots l, l+32, l+64, l+96 in order, then an xor butterfly (16,8,4,2,1); chunk totals prefix-summed in chunk order.
 *   2. u_k = ((k + w_k * 2^-32) * S) / B in float64, left to right (stratified: one draw per 1/B of the mass).
 *   3. the chunk c is the last one whose exclusive prefix is <= u_k (binary search); inside it the slots are walked in
 *      order adding to a running sum that starts at the prefix, and the first slot whose running sum exceeds u_k is
 *      drawn.  If rounding carries the walk past the chunk, the last slot of the ring with a non-zero priority is drawn
 *      (a ring whose priorities are all zero draws slot 0).  Zero-priority slots are never drawn.
 *   4. importance weights w_i = (p_min / p_i)^beta_t in float64, rounded to float (p_min: the smallest priority drawn
 *      in this batch; 1 for a slot of priority 0), kept in the workspace (dmdqn_debug_views.is_w).  The oracle
 *      (tests/replay_oracle.py) restates this order, so the drawn rows are bit-exact.
 *
 * n-step returns (hp->n_step = n > 1, any sample mode).  They assume that successive pushes of one agent are successive
 * steps in time, which is what a train loop that pushes every agent once per environment step does.  For a drawn row at
 * logical index j of agent a's ring (size sz; in prioritized mode j = (slot - (n_written - sz)) mod C; with shared
 * parameters the lookahead stays in the row's own agent's ring):
 *   m    = min(n, steps up to and including the first done at or after j, sz - j)   (the newest rows get shorter returns)
 *   z_k  = (rew[j+k] - mu) / sigma with the batch statistics of the first-step rewards (normalize_rewards), else rew[j+k]
 *   R    = z_0; g = 1; for k = 1..m-1: g = g * gamma; R = R + g * z_k   (float64, no FMA; rounded to float)
 *   the bootstrap row is j + m - 1 (its next_obs is s'), the terminal flag is its done, and the discount is 0 if it
 *   is done, else (float)(gamma^m) with gamma^m the float64 product formed left to right.
 * The workspace keeps R as r_hat, the terminal flag as the batch's dones, and the bootstrap rows and discounts
 * (dmdqn_debug_nstep).  n = 0 or 1 is the one-step target: R = r_hat, discount = (float)gamma * (1 - done), and the
 * bootstrap row is the drawn row.  n < 0 or n > DMDQN_MAX_NSTEP is refused.
 * hp->dueling other than 0 or 1 is refused here and by every other call that takes hparams. */
#define DMDQN_PER_MAX_CAPACITY (8192 * 128)
int dmdqn_sample(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                 const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                 int32_t advance_step, void* workspace, size_t workspace_bytes, void* stream);

/* Materialise the sampled batch (the five tensors ReplayBuffer.sample returns,
 * dqn_agent.py:80-85) from the workspace of the last dmdqn_sample.
 *   states, next_states device float[n_nets][batch][obs_dim] (dense, no padding)
 *   actions int32, rewards float (z-scored), dones float: device [n_nets][batch]
 *   active_out device int32[n_nets] or NULL.
 * With n-step returns (hp->n_step > 1 in dmdqn_sample) next_states are those of each row's bootstrap row, rewards are
 * the returns R and dones the terminal flags of the returns; states and actions stay those of the drawn rows. */
int dmdqn_gather(const dmdqn_dims* dims, const dmdqn_replay* replay, const void* workspace,
                 size_t workspace_bytes, float* states, int32_t* actions, float* rewards,
                 float* next_states, float* dones, int32_t* active_out, void* stream);

/* K1b + K3 + K4 -- one Double-DQN learn step for every active network.
 * Replaces DQNAgent.learn / replay (src/agents/dqn_agent.py:328-380,428-434):
 * sample, target-net forward + online argmax + TD target, online forward, MSE/Huber,
 * backward, Adam, hard/Polyak target sync.
 *   metrics_out device float[n_nets][DMDQN_METRICS_STRIDE].
 * The TD target of row i is y_i = R_i + discount_i * Q_tgt(s'_i), with s' the next_obs of the row's bootstrap row
 * (dmdqn_sample: the drawn row itself, gamma * (1 - done) and the one-step reward unless hp->n_step > 1).
 * With DMDQN_SAMPLE_PRIORITIZED the online kernel (K4a) multiplies each row's loss term and dL/dq by the row's
 * importance weight (metrics[0] is the weighted batch-mean loss; weight 1 gives the uniform path's bits) and stores
 * priority[row] = (float)pow(|q(s_i)[a_i] - y_i| + per_eps, per_alpha) (float64), raising priority_max[agent] to it
 * (atomicMax on the bits: order-independent).  A row whose priority is not finite writes nothing; nor does a row of a
 * tcgen05 K4a whose bounded waits expired.  A transition drawn twice has one delta, so both rows store the same value.
 * On the tcgen05 path the four kernels of one call form a dataflow chain (programmatic dependent launches:
 * K3 starts under the sample kernel's tail, K4a / K4b take over SMs while the previous kernel is still running
 * and wait on per-tile / per-network flags in the workspace, which the sample kernel resets).  Results are
 * bit-identical to the stage-by-stage form below; the workspace must not be shared by two calls in flight.
 * Dueling (hp->dueling = 1): before the sample kernel, a fold kernel writes W3e | b3e of the online and the target
 * network into the workspace (dmdqn_debug_dueling); K3 / K4a read the head from there, so their Q values, TD targets,
 * losses and trunk gradients are those of a plain network with the folded head.  The head update projects the folded
 * head's gradient G back onto the true parameters:
 *   dW3[k][a] = G[k][a] - (1/A) sum_{b<A} G[k][b] (a < A, else 0),  dwv[k] = sum_{b<A} G[k][b]   (likewise db3, dbv)
 * and dmdqn_learn_grads stores these at the W3 / b3 / wv / bv offsets. */
int dmdqn_learn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                float* metrics_out, void* workspace, size_t workspace_bytes, void* stream);

/* The same step, one stage per call, so a caller can bracket each kernel with CUDA events
 * (bench.py roofline): stages is a bit mask of DMDQN_STAGE_*; all four in order == dmdqn_learn (same bits;
 * kernels of different calls are ordered by the stream alone, only a call with all four stages is chained).
 * Dueling (hp->dueling = 1): the fold of the heads runs with the SAMPLE stage of this call, so the TARGET and ONLINE stages
 * need a preceding SAMPLE stage of dmdqn_learn_stages (or dmdqn_learn) on the same weights; a batch drawn by dmdqn_sample
 * leaves the folded heads of an earlier step (or none) in the workspace. */
#define DMDQN_STAGE_SAMPLE 1   /* K1b */
#define DMDQN_STAGE_TARGET 2   /* K3  */
#define DMDQN_STAGE_ONLINE 4   /* K4a */
#define DMDQN_STAGE_WGRAD  8   /* K4b */
int dmdqn_learn_stages(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                       const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                       float* metrics_out, void* workspace, size_t workspace_bytes, int32_t stages,
                       void* stream);

/* remember + replay of every agent with HOST buffers -- what the reference's train loop does per step
 * (src/scripts/train.py:274-292: agent.remember(...) then agent.replay() for every agent), as one call:
 * the step's inputs sit in ONE pinned host block (struct of arrays at the byte offsets below, each a
 * multiple of 16), which is copied to its device mirror with a single cudaMemcpyAsync; then dmdqn_push,
 * dmdqn_learn and a copy of the metrics back to host memory are queued on `stream`.  Nothing is synchronised:
 * the caller waits on the stream before reading `metrics_host` (the losses replay() returns). */
typedef struct dmdqn_step_block {
    size_t bytes;                 /* size of the host / device block */
    size_t obs_off, next_obs_off; /* float [n_agents][in_stride] */
    size_t act_off;               /* int32 [n_agents] */
    size_t rew_off;               /* double[n_agents] */
    size_t done_off;              /* uint8 [n_agents] */
    size_t draws_off;             /* [n_nets][batch] words / indices per hp->sample_mode */
    int32_t in_stride;
} dmdqn_step_block;
int dmdqn_step_host(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                    const dmdqn_nets* nets, const dmdqn_step_block* blk, const void* host_block, void* device_block,
                    float* metrics_dev, float* metrics_host, void* workspace, size_t workspace_bytes, void* stream);

/* Shared-parameter mode across ranks (n_nets == 1; not in the reference, BASELINE.json cfg5):
 * the same step but K4b stores dL/dtheta into grads_out[n_nets][layout.stride] (every float of the range the Adam calls
 * update: [0, b3 + 4), or [0, b3 + 8 + H) for dueling blocks, whose three pad floats get gradient 0) instead of
 * applying Adam, with the loss mean taken over global_batch (= batch * ranks), so that the
 * caller can sum the blocks over ranks (ncclAllReduce) and finish with dmdqn_adam_apply,
 * which takes the step's learn flags and Adam scalars (alpha_t, eps, target-sync mode) from the
 * workspace of the preceding dmdqn_learn_grads: pass it the same hparams. */
int dmdqn_learn_grads(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                      const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                      int32_t global_batch, float* grads_out, float* metrics_out, void* workspace,
                      size_t workspace_bytes, void* stream);
int dmdqn_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets,
                     const float* grads, void* workspace, size_t workspace_bytes, void* stream);

/* Global-norm gradient clipping (Keras `global_clipnorm`, tf.clip_by_global_norm, torch clip_grad_norm_): dmdqn_adam_apply
 * with every network's gradient scaled to a global norm of at most c = global_clipnorm first.  A clipped learn step is
 * dmdqn_learn_grads(..., global_batch = batch, grads, ...) followed by this call (with shared parameters across ranks: on
 * the all-reduced block, so every replica scales by the same n).  For every network g that learned this step:
 *   1. G = grads[g][0 .. layout.b3 + 4), the range dmdqn_adam_apply updates; for dueling blocks (hp->dueling = 1)
 *      [0 .. b3 + 8 + H): W3, b3, the value head wv, bv and its three pad floats;
 *   2. n = sqrt(sum G_i^2) in float64 (the squares are exact); the summation order is fixed by the kernel (8 contiguous
 *      slices, each summed by its CTA in a fixed thread order, the 8 partials added in slice order) and does not depend
 *      on the other networks or on how many networks the call covers;
 *   3. s = (float)(c / max(n, c)), the clipped gradient is G_i * s in fp32.  n <= c gives s == 1 and the update of
 *      dmdqn_adam_apply bit for bit; a non-finite n applies no scaling;
 *   4. Adam and the target sync as in dmdqn_adam_apply (the same workspace Adam scalars and the same per-element
 *      arithmetic);
 *   5. norms_out[g] (device float[n_nets], or NULL) = (float)n, the norm before clipping; 0 for a network that did not
 *      learn this step (its metrics row is 0 too).
 * A network whose step was poisoned (the workspace error flag is set: a tcgen05 kernel's bounded wait expired, so
 * metrics[g][7] < 0 and K4b wrote no gradient) gets no update and norm 0.  global_clipnorm <= 0, NaN or infinite is
 * refused with DMDQN_ERR_ARG before anything is launched. */
int dmdqn_clip_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets,
                          const float* grads, double global_clipnorm, float* norms_out, void* workspace,
                          size_t workspace_bytes, void* stream);

/* K5, shared-parameter mode over NVLink peer memory (BASELINE.json cfg5; SURVEY.md section 8 row B2/E2): ONE kernel per
 * rank that (1) announces its gradient block of this step to every peer (release store of `epoch` into the peers'
 * flag arrays), (2) waits for the peers' announcements, (3) reads every rank's block through peer pointers, sums
 * them in rank order 0..world-1 (the same order on every rank: replicas stay bit-identical) and (4) applies Adam +
 * the target sync to the local replica -- the all-reduce and the optimizer step of dmdqn_learn_grads ->
 * ncclAllReduce -> dmdqn_adam_apply in one launch, with no host round trip and no NCCL on the path.
 * grads[p] / loss[p] / flags[p] are device pointers valid on THIS device: the rank's own buffers at [rank], the
 * peers' through dmdqn_ipc_open.  The caller double-buffers grads / loss by epoch parity (a peer may already be
 * writing step t+1 while this rank still reads step t); flags[p] is uint32[DMDQN_MAX_PEERS][DMDQN_PEER_BLOCKS],
 * zero-initialised once; epoch = 1, 2, 3, ... identical on every rank.  my_loss_src is this rank's share of the loss
 * (metrics_out[0] of dmdqn_learn_grads), published to loss[rank] by the kernel; loss_out receives the sum.
 * Like dmdqn_adam_apply it takes the step's learn flag and Adam scalars from the workspace of dmdqn_learn_grads.
 * A peer that never arrives ends in DMDQN_PEER_TIMEOUT in the workspace error flag (no update applied), not in a hang. */
#define DMDQN_MAX_PEERS 8
#define DMDQN_PEER_TIMEOUT 77     /* value of the workspace error flag after a peer never arrived */
#define DMDQN_PEER_BLOCKS 128
typedef struct dmdqn_peers {
    const float* grads[DMDQN_MAX_PEERS];
    float* loss[DMDQN_MAX_PEERS];
    uint32_t* flags[DMDQN_MAX_PEERS];
    int32_t rank, world;
    uint32_t epoch;
} dmdqn_peers;
int dmdqn_allreduce_adam(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets,
                         const dmdqn_peers* peers, const float* my_loss_src, float* loss_out, void* workspace,
                         size_t workspace_bytes, void* stream);
/* CUDA IPC plumbing for the peer pointers above: export the allocation that contains dev_ptr (64-byte handle +
 * offset of dev_ptr inside it), map a peer's export on the current device (peer access is enabled lazily), unmap. */
int dmdqn_ipc_export(const void* dev_ptr, void* handle64, uint64_t* offset);
int dmdqn_ipc_open(const void* handle64, uint64_t offset, void** dev_ptr);
int dmdqn_ipc_close(void* dev_ptr, uint64_t offset);

/* Debug / parity views into the workspace after dmdqn_learn (device pointers into it):
 * y[n_nets][B], q_all[n_nets][B][4] (online Q of s), q_next[n_nets][B][4] (online Q of s'),
 * tq_all[n_nets][B][4] (target Q of s'), rows int32[n_nets][B] (agent*C + slot). */
typedef struct dmdqn_debug_views {
    const float* y; const float* q_all; const float* q_next; const float* tq_all;
    const int32_t* rows; const float* r_hat; const int32_t* active;
    const int32_t* tc_error;   /* != 0: a tcgen05 kernel's bounded mbarrier wait expired (results invalid) */
    const float* dh1; const float* dh2;   /* [n_nets][B][H] activation gradients of the last step */
    /* tcgen05 path: dh2 is never materialised; relu'(h2) as bits, uint32 [n_nets][B][H/32]
     * (bit j of word w of row i = column 32 w + j), dh2 = bit ? g_i * W3[col][a_i] : 0 */
    const uint32_t* relu2_bits;
    const float* is_w;         /* [n_nets][B] importance-sampling weights of the last prioritized sample */
} dmdqn_debug_views;
int dmdqn_debug(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_debug_views* out);
/* n-step views of the last sample (its own struct: dmdqn_debug_views keeps its size for existing callers):
 * next_rows int32[n_nets][B] (agent*C + slot of each row's bootstrap row), discount float[n_nets][B]. */
typedef struct dmdqn_nstep_views {
    const int32_t* next_rows; const float* discount;
} dmdqn_nstep_views;
int dmdqn_debug_nstep(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_nstep_views* out);
/* Dueling view of the last learn step: head float[2][n_nets][4H + 4], W3e[H][4] | b3e[4] of the online (0) and the target
 * (1) network as the fold kernel wrote them. */
typedef struct dmdqn_dueling_views {
    const float* head;
} dmdqn_dueling_views;
int dmdqn_debug_dueling(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_dueling_views* out);

/* theta_tgt <- theta for the networks whose mask is set (NULL = all).
 * Replaces DQNAgent.update_target_network (dqn_agent.py:382-384) when called explicitly. */
int dmdqn_sync_target(const dmdqn_dims* dims, const dmdqn_nets* nets, const uint8_t* mask,
                      double tau, void* stream);
/* The same on dueling parameter blocks: the whole dueling stride, value head included. */
int dmdqn_sync_target_dueling(const dmdqn_dims* dims, const dmdqn_nets* nets, const uint8_t* mask,
                              double tau, void* stream);

/* Noisy networks (Fortunato et al. 2018, factorized Gaussian noise on every layer).  The learned parameters of network g
 * are mu = nets->theta (plain or dueling layout, unchanged) and sigma, a second block of the same layout with its own
 * target copy and Adam moments.  Layer l with p inputs and q outputs (W1 / b1, W2 / b2, W3 / b3 and, for dueling blocks,
 * wv / bv) has factor vectors fin[p] and fout[q]; its weight noise is eps_ij = fin[i] * fout[j] (one fp32 product), its
 * bias noise fout[j], and the effective parameters are
 *   eff = mu + sigma * eps      (__fmul_rn, then __fadd_rn: one rounded product, one rounded sum).
 * Factor entry i of vector (layer, side) of set s (0 = online, 1 = target) at step t is f(z), f(z) = sgn(z) sqrt|z| in fp32,
 *   (x, y, -, -) = Philox4x32-10(key = {key[g] low word, high word}, counter = {i, layer << 2 | side << 1 | s, t, 0x6e6f6973})
 *   z = (float)(sqrt(-2 ln((x + 0.5) 2^-32)) cos(2 pi y 2^-32))   in float64,
 * with layer 0..3 = W1, W2, W3, the value head and side 0 = inputs, 1 = outputs.  Entries for padding are 0: W1 input rows
 * >= obs_dim, W3 output columns >= A, the value head's outputs >= 1.  t is the network's learn_step before a learn step's
 * sample kernel increments it: a learn step runs the online network (Q(s) and the double-DQN argmax at s') with set 0
 * and the target network with set 1, and acting with set 0 at the current learn_step uses the noise of the next learn
 * step's online network (the paper's rule: resample after every optimisation step).
 *   sigma, sigma_tgt, sigma_m, sigma_v  device float [n_nets][stride]  (the layout's stride)
 *   eff, eff_tgt                         device float [n_nets][stride], 16-byte aligned: written by dmdqn_noisy_fold
 *   noise                                device float [n_nets][2][record.stride]: the factor vectors of set 0 and 1
 *   key                                  device uint64 [n_nets]: each network's Philox key */
typedef struct dmdqn_noisy {
    float* sigma;
    float* sigma_tgt;
    float* sigma_m;
    float* sigma_v;
    float* eff;
    float* eff_tgt;
    float* noise;
    const uint64_t* key;
} dmdqn_noisy;

/* Float offsets of the eight factor vectors inside one set's noise record, in this order:
 *   w1_in[obs_stride] | w1_out[H] | w2_in[H] | w2_out[H] | w3_in[H] | w3_out[4] | v_in[H] | v_out[4]
 * and the record's stride (a multiple of 32 floats).  The value head's vectors are there for plain blocks too. */
typedef struct dmdqn_noise_record {
    int64_t w1_in, w1_out, w2_in, w2_out, w3_in, w3_out, v_in, v_out, stride;
} dmdqn_noise_record;
int dmdqn_noise_layout(const dmdqn_dims* dims, dmdqn_noise_record* out);

/* The factor vectors of both sets into noisy->noise and the effective blocks eff = mu + sigma * eps (set 0 from theta /
 * sigma) and eff_tgt (set 1 from theta_tgt / sigma_tgt), every float of the stride, for every network at its current
 * learn_step.  hp is read for its dueling flag only. */
int dmdqn_noisy_fold(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                     void* stream);

/* One noisy learn step up to the gradient: dmdqn_noisy_fold, then dmdqn_learn_grads with nets->theta / theta_tgt
 * replaced by eff / eff_tgt (its dueling fold, sample, K3, K4a, K4b).  grads_out receives dL/d eff; learn_step advances as
 * in dmdqn_learn_grads.  Finish the step with dmdqn_noisy_adam_apply. */
int dmdqn_learn_grads_noisy(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                            const dmdqn_nets* nets, const dmdqn_noisy* noisy, const void* draws, const uint8_t* learn_mask,
                            int32_t global_batch, float* grads_out, float* metrics_out, void* workspace,
                            size_t workspace_bytes, void* stream);

/* Adam on mu and sigma from the effective-weight gradient g of dmdqn_learn_grads_noisy: g_mu = g, g_sigma = g * eps (fp32,
 * eps of set 0 from noisy->noise), each through dmdqn_adam_apply's per-element arithmetic with the step's Adam scalars
 * (mu with adam_m / adam_v, sigma with sigma_m / sigma_v), and the target sync of both.  A network that did not learn, or
 * any network after a tcgen05 kernel set the workspace error flag, is left untouched. */
int dmdqn_noisy_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                           const float* grads, void* workspace, size_t workspace_bytes, void* stream);

/* dmdqn_act on the noisy online network at its current learn_step (set 0): the kernel streams mu and sigma and forms
 * mu + sigma * eps in registers, so q_out and the actions equal dmdqn_act / dmdqn_act_dueling on the eff block of a
 * dmdqn_noisy_fold at the same learn_step, bit for bit.  dueling: the blocks are in the dueling layout. */
int dmdqn_act_noisy(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t dueling,
                    const float* obs, int32_t obs_in_stride, const double* eps, const uint32_t* w_explore,
                    const uint32_t* w_action, int32_t* actions_out, float* q_out, void* stream);

/* dmdqn_sync_target of mu (theta -> theta_tgt) and of sigma (sigma -> sigma_tgt). */
int dmdqn_sync_target_noisy(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t dueling,
                            const uint8_t* mask, double tau, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DMDQN_B200_H */
