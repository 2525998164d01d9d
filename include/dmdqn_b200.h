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
 *   distributional networks (C51; dmdqn_param_layout_dist, see dmdqn_dist below) widen the head to 4 * Np columns:
 *     W1 | b1 | W2 | b2 | W3[H][4 * Np] | b3[4 * Np] | pad
 *   quantile networks (QR-DQN, see dmdqn_quantile below) use the same block with N quantiles in place of N atoms.
 *   implicit quantile networks (IQN, see dmdqn_iqn below) append the cosine embedding after b3:
 *     W1 | b1 | W2 | b2 | W3[H][4] | b3[4] | Wphi[n_cos][H] | bphi[H] | pad
 *   Rainbow networks (dueling noisy C51; dmdqn_param_layout_rainbow, see dmdqn_rainbow_layout below) append the per-atom
 *   value stream to the C51 block:
 *     W1 | b1 | W2 | b2 | W3[H][4 * Np] | b3[4 * Np] | Wv[H][Np] | bv[Np] | pad
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

/* Distributional Q-learning (C51, Bellemare, Dabney & Munos 2017), fp32 (FFMA) path only.  Each action's return is a
 * categorical distribution over N = n_atoms atoms (2 <= N <= 64) of the fixed support
 *   dz64 = (v_max - v_min) / (N - 1) (float64),  z_j = (float)(v_min + j * dz64),  dz = (float)dz64,
 *   lo = (float)v_min,  hi = (float)v_max                          (v_min < v_max, both finite).
 * Parameter block (dmdqn_param_layout_dist fills a dmdqn_layout):
 *   W1[obs_stride][H] | b1[H] | W2[H][H] | b2[H] | W3[H][4 * Np] | b3[4 * Np] | pad
 * with Np = N rounded up to a multiple of 4 and column a * Np + j holding atom j of action a.  Columns with a >= A or
 * j >= N are 0 and keep gradient 0.  Adam updates [0, b3 + 4 * Np); the stride is rounded up to 32 floats.
 * Head: for action a the logits are x_a = h2 . W3[:, a*Np .. a*Np + N) + b3[a*Np ..], and per action
 *   mx = max_j x_j,  e_j = expf(x_j - mx),  S = sum_j e_j (j order),  p_j = e_j / S,  log p_j = (x_j - mx) - logf(S)
 *   Q(s, a) = sum_j p_j z_j   (fmaf, j order)
 * with the accurate expf / logf and IEEE division.  Expected-Q outputs hold 0 for actions a >= A.
 * Target of sampled row i (R, discount d and the bootstrap row as dmdqn_sample forms them, so n-step returns and done
 * apply): a* = argmax of the online (double_dqn = 1) or the target (double_dqn = 0) network's expected Q at s', ties to
 * the lowest index; p = softmax of the target network's logits of a* at s'; m = 0, then for j = 0 .. N - 1 in order
 *   t = min(max(R + d * z_j, lo), hi)    (product and sum rounded separately)
 *   b = min((t - lo) / dz, N - 1),  l = floor(b),  u = ceil(b)
 *   l == u:  m[l] += p_j      else:  m[l] += p_j * (u - b);  m[u] += p_j * (b - l)
 * Loss of row i with action a_i: L_i = -sum_j m_j log p_j(s_i, a_i) (the sum as fmaf in j order, then negated); the loss
 * term is w_i * L_i with w_i the importance weight of prioritized replay (1 otherwise), and prioritized replay stores
 * priority = (float)pow(L_i + per_eps, per_alpha) (the unweighted cross-entropy).  The gradient of the logits of a_i is
 * (w_i * (p_j - m_j)) / loss_batch and 0 for every other column.  hp->loss is not read.
 * Metrics row: [0] the weighted batch-mean cross-entropy, [1] / [2] the mean and std of the online expected Q over
 * a < A, the action histogram and the learned flag.  dmdqn_debug's q_all / q_next / tq_all hold expected Q values; y is
 * not written.
 *   scratch   caller-owned device memory of at least dmdqn_dist_scratch_bytes, 16-byte aligned: the projected target
 *             distribution m [n_nets][B][Np], h2 [n_nets][B][H] and the logit gradient [n_nets][B][4 * Np].
 * Every call below refuses, before anything is launched: n_atoms outside [2, 64], v_min >= v_max or either non-finite,
 * hp->precision other than DMDQN_PRECISION_FP32, hp->dueling != 0, NULL or misaligned pointers and a scratch smaller
 * than the query returns. */
typedef struct dmdqn_dist {
    int32_t n_atoms;
    double v_min, v_max;
    void* scratch;
    size_t scratch_bytes;
} dmdqn_dist;
#define DMDQN_DIST_MAX_ATOMS 64
int dmdqn_param_layout_dist(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_layout* out);
int dmdqn_dist_scratch_bytes(const dmdqn_dims* dims, int32_t n_atoms, size_t* out_bytes);

/* One distributional learn step up to the gradient: the sample kernel of dmdqn_learn (learn_step, Adam scalars, n-step
 * and prioritized rows), then the distributional target, online and weight-gradient kernels.  grads_out[n_nets][stride]
 * receives dL/dtheta for every float of [0, b3 + 4 * Np) with the loss mean over global_batch (>= batch).  Finish the step
 * with dmdqn_adam_apply_dist. */
int dmdqn_learn_grads_dist(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_dist* dist, const dmdqn_replay* replay,
                           const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t global_batch,
                           float* grads_out, float* metrics_out, void* workspace, size_t workspace_bytes, void* stream);

/* Adam + target sync on distributional blocks from a gradient block: global_clipnorm == 0 is dmdqn_adam_apply's arithmetic,
 * global_clipnorm > 0 (finite) dmdqn_clip_adam_apply's (the norm over [0, b3 + 4 * Np), norms_out as there); a negative,
 * NaN or infinite global_clipnorm is refused. */
int dmdqn_adam_apply_dist(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, int32_t n_atoms,
                          const float* grads, double global_clipnorm, float* norms_out, void* workspace, size_t workspace_bytes,
                          void* stream);

/* dmdqn_act on distributional blocks: q_out holds the expected Q values (0 for a >= A), the action is their argmax under
 * dmdqn_act's epsilon rule, and exploring agents skip the forward pass (their q_out rows are untouched).  dist->scratch is
 * not used and may be NULL. */
int dmdqn_act_dist(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_dist* dist, const float* obs,
                   int32_t obs_in_stride, const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
                   int32_t* actions_out, float* q_out, void* stream);

/* dmdqn_sync_target over the whole distributional stride. */
int dmdqn_sync_target_dist(const dmdqn_dims* dims, const dmdqn_nets* nets, int32_t n_atoms, const uint8_t* mask, double tau,
                           void* stream);

/* The scratch's views after dmdqn_learn_grads_dist: target_dist float[n_nets][B][Np] (the projected m of every row),
 * h2 float[n_nets][B][H], dlogits float[n_nets][B][4 * Np] (the logit gradient). */
typedef struct dmdqn_dist_views {
    const float* target_dist; const float* h2; const float* dlogits;
} dmdqn_dist_views;
int dmdqn_debug_dist(const dmdqn_dims* dims, const dmdqn_dist* dist, dmdqn_dist_views* out);

/* Quantile regression DQN (QR-DQN, Dabney, Rowland, Bellemare & Munos 2018), fp32 (FFMA) path only.  Each action's
 * return is N = n_quantiles quantiles (2 <= N <= DMDQN_DIST_MAX_ATOMS) at the fixed midpoints
 *   tau_i = (float)((2 i + 1) / (2.0 N))   (float64 division, then rounded)
 * and the values of the quantiles are learned, so there is no support to choose.  The parameter block, its padding and
 * the Adam range are those of dmdqn_dist with N atoms (dmdqn_param_layout_dist(dims, N)); column a * Np + i holds
 * quantile i of action a.  After the head, every operation below is one rounded fp32 operation unless stated, and none
 * is fused (no FMA).
 * Head: theta_{a,i}(s) = h2 . W3[:, a*Np + i] + b3[a*Np + i] (the C51 logits, computed as C51 computes them), and
 *   Q(s, a) = (sum_i theta_{a,i}, adds in i order from 0) / (float)N      (IEEE division; 0 for actions a >= A)
 * Target of sampled row r (R, discount d and the bootstrap row as dmdqn_sample forms them, so n-step returns and done
 * apply): a* = argmax of the online (double_dqn = 1) or the target (double_dqn = 0) network's Q at s', ties to the
 * lowest index, and for j < N
 *   T_j = R + d * theta^tgt_{a*, j}(s')   (product and sum rounded separately; not differentiated)
 * Loss of row r with action a_r, k = (float)kappa: for each pair (i, j), theta_i = theta_{a_r,i}(s),
 *   u = T_j - theta_i,  w = u < 0 ? 1 - tau_i : tau_i
 *   k > 0:  rho = w * (|u| <= k ? (0.5 * (u * u)) / k : |u| - 0.5 * k),   drho = (-w * min(max(u, -k), k)) / k
 *   k = 0:  rho = w * |u|,   drho = u > 0 ? -w : u < 0 ? w : 0
 *   L_r = (sum_i (sum_j rho_ij, j order) in i order) / (float)N,   g_i = (sum_j drho_ij, j order) / (float)N
 * every sum an fp32 add from 0.  The loss term is w_r * L_r with w_r the importance weight of prioritized replay (1
 * otherwise), prioritized replay stores priority = (float)pow(L_r + per_eps, per_alpha) (the unweighted loss), and the
 * gradient of column a_r * Np + i is (w_r * g_i) / loss_batch (0 for i >= N and for every other action's columns).
 * hp->loss is not read.
 * Metrics row: [0] the weighted batch-mean loss, [1] / [2] the mean and std of the online Q over a < A, the action
 * histogram and the learned flag.  dmdqn_debug's q_all / q_next / tq_all hold expected Q values; y is not written.
 *   kappa     the Huber threshold: finite and >= 0; 0 is the pure quantile loss (QR-DQN-0).
 *   scratch   caller-owned device memory of at least dmdqn_dist_scratch_bytes(dims, N), 16-byte aligned, with the regions
 *             of dmdqn_dist: the target samples T [n_nets][B][Np] (0 for j >= N), h2 and the logit gradient.
 * Every call below refuses, before anything is launched: n_quantiles outside [2, 64], kappa negative, NaN or infinite,
 * hp->precision other than DMDQN_PRECISION_FP32, hp->dueling != 0, NULL or misaligned pointers and a scratch smaller
 * than the query returns.  Adam, clipping and the target sync are dmdqn_adam_apply_dist and dmdqn_sync_target_dist with
 * n_atoms = N. */
typedef struct dmdqn_quantile {
    int32_t n_quantiles;
    double kappa;
    void* scratch;
    size_t scratch_bytes;
} dmdqn_quantile;

/* One quantile learn step up to the gradient: the sample kernel of dmdqn_learn (learn_step, Adam scalars, n-step and
 * prioritized rows), then the quantile target, online and (C51) weight-gradient kernels.  grads_out[n_nets][stride]
 * receives dL/dtheta for every float of [0, b3 + 4 * Np) with the loss mean over global_batch (>= batch).  Finish the step
 * with dmdqn_adam_apply_dist(..., N, ...). */
int dmdqn_learn_grads_quantile(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_quantile* quantile,
                               const dmdqn_replay* replay, const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                               int32_t global_batch, float* grads_out, float* metrics_out, void* workspace,
                               size_t workspace_bytes, void* stream);

/* dmdqn_act on quantile blocks: q_out holds the expected Q values (0 for a >= A), the action is their argmax under
 * dmdqn_act's epsilon rule, and exploring agents skip the forward pass (their q_out rows are untouched).
 * quantile->scratch and kappa are not used; the scratch may be NULL. */
int dmdqn_act_quantile(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_quantile* quantile, const float* obs,
                       int32_t obs_in_stride, const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
                       int32_t* actions_out, float* q_out, void* stream);

/* The scratch's views after dmdqn_learn_grads_quantile: target_dist holds the target samples T [n_nets][B][Np]; h2 and
 * dlogits are as in dmdqn_debug_dist. */
int dmdqn_debug_quantile(const dmdqn_dims* dims, const dmdqn_quantile* quantile, dmdqn_dist_views* out);

/* Implicit quantile networks (IQN, Dabney, Ostrovski, Silver & Munos 2018), fp32 (FFMA) path only.  The network takes a
 * quantile fraction tau as an input and returns the return quantile Z_tau(s, a).  Layer 1 is the state embedding and layer 2
 * plus the head are the function of the product:
 *   h1       = relu(s W1 + b1)                                     (once per row)
 *   c_m(tau) = (float)cos(M_PI * m * (double)tau),  m = 0 .. n_cos - 1   (float64, then rounded)
 *   phi(tau) = relu(c(tau) Wphi + bphi)
 *   z        = h1 * phi(tau)                                       (one fp32 product per element)
 *   h2       = relu(z W2 + b2)
 *   Z_tau(s, a) = h2 . W3[:, a] + b3[a]                            (the plain 4-wide head; 0 for a >= A)
 * Parameter block (dmdqn_param_layout_iqn):
 *   W1 | b1 | W2 | b2 | W3[H][4] | b3[4] | Wphi[n_cos][H] | bphi[H] | pad
 * with the plain offsets up to b3 and Wphi at b3 + 4 (16-byte aligned); Adam updates [0, end = bphi + H); the stride is
 * rounded up to 32 floats.
 * Fractions, drawn on the device: fraction i of sampled row r of network g, set 0 (tau_i, i < N) or 1 (tau'_j, j < N'), is
 *   (x, -, -, -) = Philox4x32-10(key = {key[g] low word, high word}, counter = {row_base + r, i, t, 0x69716e00 | set})
 *   tau = ((x >> 9) + 0.5) * 2^-23       (the top 23 bits, exact in fp32, strictly inside (0, 1))
 * with t the network's learn_step before the sample kernel increments it (the noisy networks' rule) and row_base the global
 * index of the caller's first row (0 in one process, rank * B when ranks split a shared batch).
 * Policy: Q(s, a) = (sum_k Z_{tau~_k}(s, a), k order) / (float)K at the K midpoints tau~_k = (float)((2k + 1) / (2.0 K)).  (The
 * paper draws K random fractions; the midpoint rule estimates the same integral and makes acting deterministic.)  a* is the
 * argmax of the online (double_dqn = 1) or the target (double_dqn = 0) network's Q at s', ties to the lowest index.
 * Target samples T_j = R + d * Z^tgt_{tau'_j}(s', a*) (product and sum rounded separately; R, d and the bootstrap row as
 * dmdqn_sample forms them).  With theta_i = Z_{tau_i}(s, a_r), rho_ij and drho_ij are dmdqn_quantile's pair terms with w taken
 * from the sampled tau_i, and
 *   L_r = (sum_i (sum_j rho_ij, j order), i order) / (float)N',   g_i = (sum_j drho_ij, j order) / (float)N'
 * (with N = N' and the midpoints as tau_i these are QR-DQN's formulas).  The loss term is w_r * L_r, the gradient of
 * Z_{tau_i}(s, a_r) is (w_r * g_i) / loss_batch, and prioritized replay stores (float)pow(L_r + per_eps, per_alpha)
 * (a transition drawn by several rows of the batch gets the priority of its last row: the rows' fractions differ).
 * hp->loss is not read.  The backward pass runs through the head, layer 2 (dz = dh2 W2^T), the product (dphi = dz * h1 masked
 * by relu'(phi); dh1 = (sum_i dz_i * phi_i, i order) masked by relu'(h1)) and both embeddings.
 * Metrics row: [0] the weighted batch-mean loss, [1] / [2] the mean and std over a < A of the online Q at s taken as the
 * SAMPLE mean over the N fractions tau_i (not the K-midpoint Q), the action histogram and the learned flag.  dmdqn_debug's
 * q_all holds those sample means, q_next the K-midpoint Q of the network that picks a*, tq_all the mean of the N' sampled
 * target values of every action; y is not written.
 *   n_tau N, n_tau_prime N', n_policy K   each in [1, DMDQN_IQN_MAX_TAU]
 *   n_cos      a multiple of 4 in [4, DMDQN_IQN_MAX_COS]
 *   kappa      the Huber threshold: finite and >= 0
 *   row_base   >= 0
 *   key        device uint64 [n_nets]: each network's Philox key (read by the learn call only)
 *   scratch    caller-owned device memory of at least dmdqn_iqn_scratch_bytes, 16-byte aligned (learn and debug only)
 * Every call below refuses, before anything is launched: counts outside their range, a bad n_cos, kappa negative, NaN or
 * infinite, row_base < 0, hp->precision other than DMDQN_PRECISION_FP32, hp->dueling != 0, NULL or misaligned pointers (a
 * NULL key for learn) and a short scratch. */
typedef struct dmdqn_iqn {
    int32_t n_tau, n_tau_prime, n_policy, n_cos;
    double kappa;
    int64_t row_base;
    const uint64_t* key;
    void* scratch;
    size_t scratch_bytes;
} dmdqn_iqn;
#define DMDQN_IQN_MAX_TAU 64
#define DMDQN_IQN_MAX_COS 128

typedef struct dmdqn_iqn_layout {
    int64_t w1, b1, w2, b2, w3, b3, wphi, bphi, end, stride;
} dmdqn_iqn_layout;
int dmdqn_param_layout_iqn(const dmdqn_dims* dims, int32_t n_cos, dmdqn_iqn_layout* out);
int dmdqn_iqn_scratch_bytes(const dmdqn_dims* dims, const dmdqn_iqn* iqn, size_t* out_bytes);

/* One IQN learn step up to the gradient: the sample kernel of dmdqn_learn (learn_step, Adam scalars, n-step and prioritized
 * rows), then iqn_target_kernel, iqn_online_kernel and iqn_wgrad_kernel.  grads_out[n_nets][stride] receives dL/dtheta for
 * every float of [0, end) with the loss mean over global_batch (>= batch).  Finish with dmdqn_adam_apply_iqn. */
int dmdqn_learn_grads_iqn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_iqn* iqn, const dmdqn_replay* replay,
                          const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t global_batch,
                          float* grads_out, float* metrics_out, void* workspace, size_t workspace_bytes, void* stream);

/* Adam + target sync on IQN blocks, as dmdqn_adam_apply_dist: global_clipnorm == 0 is dmdqn_adam_apply's arithmetic,
 * global_clipnorm > 0 (finite) dmdqn_clip_adam_apply's with the norm over [0, end) (Wphi and bphi included). */
int dmdqn_adam_apply_iqn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, int32_t n_cos,
                         const float* grads, double global_clipnorm, float* norms_out, void* workspace, size_t workspace_bytes,
                         void* stream);

/* dmdqn_act on IQN blocks: q_out holds the K-midpoint Q (0 for a >= A), the action is its argmax under dmdqn_act's epsilon
 * rule, and exploring agents skip the forward pass (their q_out rows are untouched).  iqn->key, kappa, row_base, n_tau,
 * n_tau_prime and the scratch are not used. */
int dmdqn_act_iqn(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_iqn* iqn, const float* obs, int32_t obs_in_stride,
                  const double* eps, const uint32_t* w_explore, const uint32_t* w_action, int32_t* actions_out, float* q_out,
                  void* stream);

/* dmdqn_sync_target over the whole IQN stride. */
int dmdqn_sync_target_iqn(const dmdqn_dims* dims, const dmdqn_nets* nets, int32_t n_cos, const uint8_t* mask, double tau,
                          void* stream);

/* The scratch's views after dmdqn_learn_grads_iqn: tau [n_nets][B][N], tau_prime [n_nets][B][N'], target (T) [n_nets][B][N'],
 * theta [n_nets][B][N] (the online values of the taken action), grad [n_nets][B][N] ((w_r g_i) / loss_batch), and the
 * activation gradients of every (row, fraction) at s, fraction-major: dh2 and dphi [n_nets][N][B][H] (dmdqn_debug's dh1
 * holds dh1 [n_nets][B][H]). */
typedef struct dmdqn_iqn_views {
    const float* tau; const float* tau_prime; const float* target; const float* theta; const float* grad;
    const float* dh2; const float* dphi;
} dmdqn_iqn_views;
int dmdqn_debug_iqn(const dmdqn_dims* dims, const dmdqn_iqn* iqn, dmdqn_iqn_views* out);

/* Rainbow (Hessel et al. 2018): C51 heads (dmdqn_dist) with dueling value / advantage streams and noisy layers everywhere
 * (dmdqn_noisy), fp32 (FFMA) path only.  Prioritized replay, n-step returns and double DQN apply as for every learn step.
 * Parameter block (dmdqn_param_layout_rainbow):
 *   W1 | b1 | W2 | b2 | W3[H][4 * Np] | b3[4 * Np] | Wv[H][Np] | bv[Np] | pad
 * with the C51 offsets up to b3, wv at the C51 end (b3 + 4 * Np, 16-byte aligned), bv = wv + H * Np, end = bv + Np (Adam
 * updates [0, end)) and the stride rounded up to 32 floats.  Value columns j >= N are 0 and keep gradient 0, as do the C51
 * pad columns.  The logits x_{a,j} = V_j + Adv_{a,j} - (1/A) sum_{b<A} Adv_{b,j} are linear in h2, so the head folds per atom:
 * for every row k < H, and the bias row (b3 / bv), and every j < N
 *   W3e[k][a * Np + j] = head_fold({W3[k][b * Np + j]}_{b<4}, Wv[k][j], A)[a]      (dmdqn_hparams.dueling's fold, per atom)
 * and columns j >= N or a >= A of W3e | b3e are 0.  After the fold the step is dmdqn_dist's on W3e | b3e: softmax, expected Q,
 * projection, cross-entropy, priority and metrics row.  With G the gradient with respect to W3e | b3e, the head update is
 * head_project per (k, j): the advantage gradient {dW3[k][a * Np + j]}_a = G[k][a * Np + j] - (1/A) sum_{b<A} G[k][b * Np + j]
 * (0 for a >= A) and dWv[k][j] = sum_{b<A} G[k][b * Np + j] (likewise b3 / bv; 0 for j >= N).
 * Noise: dmdqn_noisy's rule with the Rainbow record (dmdqn_noise_layout_rainbow; the same struct)
 *   w1_in[obs_stride] | w1_out[H] | w2_in[H] | w2_out[H] | w3_in[H] | w3_out[4 * Np] | v_in[H] | v_out[Np]
 * (stride a multiple of 32): output factor i of w3_out is column a * Np + j, 0 unless a < A and j < N; v_out[j] is 0 for
 * j >= N.  The Philox counters, Box-Muller, eps = fin[k] * fout[col] for a weight and fout[col] for a bias, and
 * eff = mu + sigma * eps are dmdqn_noisy's.
 * A learn step runs, in order: 1. the noise fold (sets 0 and 1 at the learn_step t before the increment, into eff / eff_tgt);
 * 2. the head fold of eff (online) and eff_tgt (target) into the scratch; 3. the sample kernel; 4. the C51 target and online
 * kernels on the folded heads with the eff trunks; 5. the C51 weight-gradient kernel; 6. the projection, which leaves dL/d eff
 * in the Rainbow layout in grads_out; then dmdqn_adam_apply_rainbow: 7. Adam on mu (g) and sigma (g * eps of set 0) and the
 * target sync of both.  Acting uses set 0 at the current learn_step (the noisy rule); greedy evaluation uses mu alone.
 *   dist       dmdqn_dist (n_atoms, support); its scratch holds at least dmdqn_rainbow_scratch_bytes, 16-byte aligned: the C51
 *              regions, then the folded heads float [2][n_nets][(H + 1) * 4 * Np] (W3e | b3e, online then target).
 *   noisy      dmdqn_noisy over Rainbow blocks; noise is [n_nets][2][record stride] of the Rainbow record.
 * Every call below refuses, before anything is launched: n_atoms outside [2, 64], a bad support, hp->precision other than
 * DMDQN_PRECISION_FP32, hp->dueling != 1 (calls that take hparams: Rainbow blocks always carry the value stream), NULL or
 * misaligned pointers (every dmdqn_noisy field for learn, Adam and the target sync) and a short scratch. */
typedef struct dmdqn_rainbow_layout {
    int64_t w1, b1, w2, b2, w3, b3, wv, bv, end, stride;
} dmdqn_rainbow_layout;
int dmdqn_param_layout_rainbow(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_rainbow_layout* out);
int dmdqn_noise_layout_rainbow(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_noise_record* out);
int dmdqn_rainbow_scratch_bytes(const dmdqn_dims* dims, int32_t n_atoms, size_t* out_bytes);

/* Steps 1 and 2 at every network's current learn_step: the factor vectors into noisy->noise, eff / eff_tgt, and the folded
 * heads into dist->scratch. */
int dmdqn_rainbow_fold(const dmdqn_dims* dims, const dmdqn_dist* dist, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                       void* stream);

/* Steps 1 to 6: grads_out[n_nets][stride] receives dL/d eff for every float of [0, end) with the loss mean over global_batch
 * (>= batch); learn_step advances as in dmdqn_learn_grads.  Finish the step with dmdqn_adam_apply_rainbow. */
int dmdqn_learn_grads_rainbow(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_dist* dist,
                              const dmdqn_replay* replay, const dmdqn_nets* nets, const dmdqn_noisy* noisy, const void* draws,
                              const uint8_t* learn_mask, int32_t global_batch, float* grads_out, float* metrics_out,
                              void* workspace, size_t workspace_bytes, void* stream);

/* Step 7, as dmdqn_noisy_adam_apply over [0, end) of Rainbow blocks. */
int dmdqn_adam_apply_rainbow(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                             int32_t n_atoms, const float* grads, void* workspace, size_t workspace_bytes, void* stream);

/* dmdqn_act_dist on Rainbow blocks, the head folded per atom in registers.  noisy set: mu + sigma * eps with set 0's noise at
 * the current learn_step, so q_out and the actions equal dmdqn_act_dist's on the C51 block that holds eff's trunk and its
 * folded head after a dmdqn_rainbow_fold at the same learn_step, bit for bit.  noisy NULL: mu alone (greedy evaluation).
 * dist->scratch is not used and may be NULL. */
int dmdqn_act_rainbow(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, const dmdqn_dist* dist,
                      const float* obs, int32_t obs_in_stride, const double* eps, const uint32_t* w_explore,
                      const uint32_t* w_action, int32_t* actions_out, float* q_out, void* stream);

/* dmdqn_sync_target over the whole Rainbow stride, of mu (theta -> theta_tgt) and of sigma (sigma -> sigma_tgt). */
int dmdqn_sync_target_rainbow(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t n_atoms,
                              const uint8_t* mask, double tau, void* stream);

/* The scratch's views after dmdqn_learn_grads_rainbow (or dmdqn_rainbow_fold, for head): dmdqn_dist_views, and head float
 * [2][n_nets][(H + 1) * 4 * Np], the folded W3e | b3e of the online (0) and the target (1) network. */
typedef struct dmdqn_rainbow_views {
    const float* target_dist; const float* h2; const float* dlogits; const float* head;
} dmdqn_rainbow_views;
int dmdqn_debug_rainbow(const dmdqn_dims* dims, const dmdqn_dist* dist, dmdqn_rainbow_views* out);

#ifdef __cplusplus
}
#endif
#endif /* DMDQN_B200_H */
