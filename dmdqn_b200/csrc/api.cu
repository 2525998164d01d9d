// extern "C" surface of libdmdqn_b200.so (include/dmdqn_b200.h): argument validation and
// dispatch only; the kernels live in featurize.cu, act.cu, replay.cu and learn.cu.
#include <stdarg.h>
#include <string.h>
#include "common.cuh"

namespace dmdqn {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int validate_dims(const dmdqn_dims* d) {
    DMDQN_CHECK_ARG(d != nullptr, "dims is NULL");
    DMDQN_CHECK_ARG(d->n_agents >= 1, "n_agents=%d must be >= 1", d->n_agents);
    DMDQN_CHECK_ARG(d->n_nets == d->n_agents || d->n_nets == 1,
                    "n_nets=%d must be n_agents (independent) or 1 (shared)", d->n_nets);
    DMDQN_CHECK_ARG(d->obs_dim >= 1 && d->obs_stride >= d->obs_dim && d->obs_stride % 16 == 0 &&
                        d->obs_stride <= 128,
                    "obs_dim=%d obs_stride=%d: stride must be a multiple of 16 in [obs_dim, 128]",
                    d->obs_dim, d->obs_stride);
    DMDQN_CHECK_ARG(d->hidden == 64 || d->hidden == 128 || d->hidden == 256 || d->hidden == 512,
                    "hidden=%d: supported widths are 64, 128, 256, 512 (nn_layers=[H,H])", d->hidden);
    DMDQN_CHECK_ARG(d->n_actions >= 1 && d->n_actions <= DMDQN_MAX_ACTIONS, "n_actions=%d must be in [1,4]",
                    d->n_actions);
    DMDQN_CHECK_ARG(d->batch >= 1 && d->batch <= 4096, "batch=%d must be in [1,4096]", d->batch);
    DMDQN_CHECK_ARG(d->capacity >= 1, "capacity=%d must be >= 1", d->capacity);
    DMDQN_CHECK_ARG((int64_t)d->n_agents * d->capacity < (int64_t)1 << 31,
                    "n_agents*capacity=%lld overflows the int32 row id",
                    (long long)d->n_agents * d->capacity);
    return DMDQN_OK;
}

int device_sm_count(int* n_sm) {
    static int cache[kMaxDevices] = {};
    int dev = 0;
    DMDQN_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices || !cache[dev]) {
        int n = 0;
        DMDQN_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        if (dev >= 0 && dev < kMaxDevices) cache[dev] = n;
        *n_sm = n;
        return DMDQN_OK;
    }
    *n_sm = cache[dev];
    return DMDQN_OK;
}

int opt_in_dynamic_smem(const void* kernel, size_t bytes, size_t (&cache)[kMaxDevices]) {
    if (bytes <= 48 * 1024) return DMDQN_OK;
    int dev = 0;
    DMDQN_CUDA(cudaGetDevice(&dev));
    const bool cached = dev >= 0 && dev < kMaxDevices;
    if (cached && cache[dev] >= bytes) return DMDQN_OK;
    DMDQN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (cached) cache[dev] = bytes;
    return DMDQN_OK;
}

static int check_workspace(const dmdqn_dims* dims, void* ws, size_t bytes, Workspace* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    *out = make_workspace(*dims);
    DMDQN_CHECK_ARG(ws != nullptr, "workspace is NULL");
    if (bytes < out->total) {
        set_error("workspace has %zu bytes, %zu needed", bytes, out->total);
        return DMDQN_ERR_WORKSPACE;
    }
    return DMDQN_OK;
}

}  // namespace dmdqn

using namespace dmdqn;

// The offsets every public layout struct shares
template <class T>
static void copy_trunk(const Layout& l, T* out) {
    out->w1 = l.w1; out->b1 = l.b1; out->w2 = l.w2; out->b2 = l.b2;
    out->w3 = l.w3; out->b3 = l.b3; out->stride = l.stride;
}

static void copy_noise_rec(const NoiseRec& r, dmdqn_noise_record* out) {
    int64_t* f[8] = {&out->w1_in, &out->w1_out, &out->w2_in, &out->w2_out, &out->w3_in, &out->w3_out, &out->v_in, &out->v_out};
    for (int v = 0; v < 8; ++v) *f[v] = r.off[v];
    out->stride = r.stride;
}

// Adam over the block of head shape hs, after global-norm clipping when clipnorm > 0
static int run_adam(const dmdqn_dims& d, const dmdqn_hparams& hp, HeadShape hs, const dmdqn_nets& nets, const float* grads,
                    double clipnorm, float* norms_out, void* workspace, const Workspace& w, void* stream) {
    const LearnArgs A = make_learn_args(d, hp, hs, {}, nets, (char*)workspace, w, nullptr, nullptr, 0);
    return launch_adam(A, grads, clipnorm, norms_out, (cudaStream_t)stream);
}

// The target sync of a noisy block: mu, then sigma
static int sync_noisy(const dmdqn_dims& d, HeadShape hs, const dmdqn_nets& nets, const dmdqn_noisy& nz, const uint8_t* mask,
                      double tau, void* stream) {
    const int64_t stride = make_layout(d.obs_stride, d.hidden, hs).stride;
    if (int rc = launch_sync_target(d, stride, nets.theta, nets.theta_tgt, mask, tau, (cudaStream_t)stream)) return rc;
    return launch_sync_target(d, stride, nz.sigma, nz.sigma_tgt, mask, tau, (cudaStream_t)stream);
}

extern "C" {

const char* dmdqn_last_error(void) { return g_error; }
int dmdqn_abi_version(void) { return DMDQN_ABI_VERSION; }

int dmdqn_param_layout(const dmdqn_dims* dims, dmdqn_layout* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    copy_trunk(make_layout(dims->obs_stride, dims->hidden), out);
    return DMDQN_OK;
}

int dmdqn_param_layout_dueling(const dmdqn_dims* dims, dmdqn_dueling_layout* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const Layout l = make_layout(dims->obs_stride, dims->hidden, {1, 1, true, 0});
    copy_trunk(l, out);
    out->wv = l.wv; out->bv = l.bv;
    return DMDQN_OK;
}

int dmdqn_workspace_bytes(const dmdqn_dims* dims, size_t* out_bytes) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out_bytes != nullptr, "out_bytes is NULL");
    *out_bytes = make_workspace(*dims).total;
    return DMDQN_OK;
}

int dmdqn_featurize(int32_t n, const int32_t* halting, const int32_t* phase, const double* next_switch,
                    const double* phase_dur, double sim_time, const uint8_t* signal_valid,
                    const int32_t* nbr_idx, const int32_t* phase_lut, const double* snapshot,
                    double local_weight, double global_weight, double* own_out, float* obs_out,
                    int32_t obs_out_stride, double* reward_out, double* global_out, int64_t* scratch,
                    void* stream) {
    DMDQN_CHECK_ARG(n >= 1, "n=%d must be >= 1", n);
    DMDQN_CHECK_ARG(halting && phase && next_switch && phase_dur && signal_valid && nbr_idx && phase_lut,
                    "featurize: NULL input");
    DMDQN_CHECK_ARG(obs_out && reward_out && global_out && scratch, "featurize: NULL output");
    DMDQN_CHECK_ARG(obs_out_stride >= DMDQN_OBS_DIM, "obs_out_stride=%d must be >= 89", obs_out_stride);
    return launch_featurize(n, halting, phase, next_switch, phase_dur, sim_time, signal_valid, nbr_idx,
                            phase_lut, snapshot, local_weight, global_weight, own_out, obs_out,
                            obs_out_stride, reward_out, global_out, scratch, (cudaStream_t)stream);
}

int dmdqn_featurize_alt(int32_t n, const int32_t* halting, const int32_t* phase, const double* next_switch,
                        const uint8_t* signal_valid, double sim_time, const int32_t* nbr_idx, const double* prev_own,
                        double* own_out, float* obs_out, int32_t obs_out_stride, double* reward_out, void* stream) {
    DMDQN_CHECK_ARG(n >= 1, "n=%d must be >= 1", n);
    DMDQN_CHECK_ARG(halting && phase && next_switch && signal_valid && nbr_idx, "featurize_alt: NULL input");
    DMDQN_CHECK_ARG(obs_out != nullptr, "featurize_alt: obs_out is NULL");
    DMDQN_CHECK_ARG(obs_out_stride >= DMDQN_OBS_ALT_DIM, "obs_out_stride=%d must be >= 74", obs_out_stride);
    return launch_featurize_alt(n, halting, phase, next_switch, signal_valid, sim_time, nbr_idx, prev_own, own_out,
                                obs_out, obs_out_stride, reward_out, (cudaStream_t)stream);
}

static int run_act(const dmdqn_dims* dims, const dmdqn_nets* nets, const float* obs, int32_t obs_in_stride,
                   const double* eps, const uint32_t* w_explore, const uint32_t* w_action, int32_t* actions_out,
                   float* q_out, bool dueling, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && obs && eps && w_explore && w_action && actions_out, "act: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act(*dims, *nets, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out, dueling,
                      (cudaStream_t)stream);
}

int dmdqn_act(const dmdqn_dims* dims, const dmdqn_nets* nets, const float* obs, int32_t obs_in_stride,
              const double* eps, const uint32_t* w_explore, const uint32_t* w_action, int32_t* actions_out,
              float* q_out, void* stream) {
    return run_act(dims, nets, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out, false, stream);
}

int dmdqn_act_dueling(const dmdqn_dims* dims, const dmdqn_nets* nets, const float* obs, int32_t obs_in_stride,
                      const double* eps, const uint32_t* w_explore, const uint32_t* w_action, int32_t* actions_out,
                      float* q_out, void* stream) {
    return run_act(dims, nets, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out, true, stream);
}

int dmdqn_push(const dmdqn_dims* dims, const dmdqn_replay* replay, const float* obs, const int32_t* act,
               const double* rew, const float* next_obs, const uint8_t* done, int32_t in_stride,
               const uint8_t* mask, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(replay && replay->obs && replay->next_obs && replay->act && replay->rew && replay->done &&
                        replay->n_written, "push: NULL replay pointer");
    DMDQN_CHECK_ARG(!replay->priority || replay->priority_max, "push: priority is set but priority_max is NULL");
    DMDQN_CHECK_ARG(obs && act && rew && next_obs && done, "push: NULL transition pointer");
    DMDQN_CHECK_ARG(in_stride >= dims->obs_dim, "in_stride=%d < obs_dim=%d", in_stride, dims->obs_dim);
    return launch_push(*dims, *replay, obs, act, rew, next_obs, done, in_stride, mask, (cudaStream_t)stream);
}

static int check_n_step(const dmdqn_hparams* hp) {
    DMDQN_CHECK_ARG(hp->n_step >= 0 && hp->n_step <= DMDQN_MAX_NSTEP, "n_step=%d must be in [0, %d] (0 and 1: one-step targets)",
                    hp->n_step, DMDQN_MAX_NSTEP);
    return DMDQN_OK;
}

static_assert(offsetof(dmdqn_hparams, dueling) == 76 && sizeof(dmdqn_hparams) == 112,
              "dueling sits in the former interior padding of dmdqn_hparams: no other field moves");

static int check_dueling(const dmdqn_hparams* hp) {
    DMDQN_CHECK_ARG(hp->dueling == 0 || hp->dueling == 1, "dueling=%d must be 0 (plain head) or 1 (dueling heads)", hp->dueling);
    return DMDQN_OK;
}

static int check_learn_args(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                            const dmdqn_nets* nets, const void* draws) {
    DMDQN_CHECK_ARG(hp && replay && nets && draws, "NULL argument");
    if (int rc = check_n_step(hp)) return rc;
    if (int rc = check_dueling(hp)) return rc;
    DMDQN_CHECK_ARG(replay->obs && replay->next_obs && replay->act && replay->rew && replay->done &&
                        replay->n_written, "NULL replay pointer");
    DMDQN_CHECK_ARG(nets->theta && nets->theta_tgt && nets->adam_m && nets->adam_v && nets->learn_step,
                    "NULL network pointer");
    DMDQN_CHECK_ARG(hp->sample_mode >= 0 && hp->sample_mode <= DMDQN_SAMPLE_PRIORITIZED, "sample_mode=%d", hp->sample_mode);
    if (hp->sample_mode == DMDQN_SAMPLE_PRIORITIZED) {
        DMDQN_CHECK_ARG(replay->priority && replay->priority_max,
                        "sample_mode=prioritized needs the replay's priority and priority_max arrays (NULL priority pointer)");
        DMDQN_CHECK_ARG(!(dims->n_nets == 1 && dims->n_agents > 1),
                        "sample_mode=prioritized serves independent networks only (n_nets=%d, n_agents=%d share parameters)",
                        dims->n_nets, dims->n_agents);
    }
    DMDQN_CHECK_ARG(hp->loss == DMDQN_LOSS_MSE || hp->loss == DMDQN_LOSS_HUBER, "loss=%d", hp->loss);
    DMDQN_CHECK_ARG(hp->precision >= DMDQN_PRECISION_FP32 && hp->precision <= DMDQN_PRECISION_TF32X3, "precision=%d",
                    hp->precision);
    return DMDQN_OK;
}

// Validation, the sample kernel (when `stages` has it) and the learn kernels of one step.  grads != NULL: K4b stores
// dL/dtheta there instead of applying Adam, with the loss mean over global_batch.
static int run_learn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay, const dmdqn_nets* nets,
                     const void* draws, const uint8_t* learn_mask, float* metrics_out, void* workspace,
                     size_t workspace_bytes, int32_t stages, float* grads, int32_t global_batch, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    rc = check_learn_args(dims, hp, replay, nets, draws);
    if (rc) return rc;
    if (grads) DMDQN_CHECK_ARG(global_batch >= dims->batch, "global_batch=%d < batch=%d", global_batch, dims->batch);
    if (stages & DMDQN_STAGE_SAMPLE) {
        if (hp->dueling) {            // W3e | b3e of this step's weights, complete before the sample -> K3 -> K4a -> K4b chain
            rc = launch_head_fold(*dims, {1, 1, true, 0}, nets->theta, nets->theta_tgt,
                                  reinterpret_cast<float*>((char*)workspace + w.head), (cudaStream_t)stream);
            if (rc) return rc;
        }
        rc = launch_sample(*dims, *hp, *replay, *nets, draws, learn_mask, 1, (char*)workspace, w, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return launch_learn(*dims, *hp, *replay, *nets, metrics_out, (char*)workspace, w, stages, grads, global_batch,
                        (cudaStream_t)stream);
}

int dmdqn_sample(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                 const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t advance_step,
                 void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    rc = check_learn_args(dims, hp, replay, nets, draws);
    if (rc) return rc;
    return launch_sample(*dims, *hp, *replay, *nets, draws, learn_mask, advance_step, (char*)workspace, w,
                         (cudaStream_t)stream);
}

int dmdqn_gather(const dmdqn_dims* dims, const dmdqn_replay* replay, const void* workspace,
                 size_t workspace_bytes, float* states, int32_t* actions, float* rewards, float* next_states,
                 float* dones, int32_t* active_out, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, const_cast<void*>(workspace), workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(replay && replay->obs && replay->next_obs, "gather: NULL replay pointer");
    DMDQN_CHECK_ARG(states && actions && rewards && next_states && dones, "gather: NULL output");
    return launch_gather(*dims, *replay, (const char*)workspace, w, states, actions, rewards, next_states, dones,
                         active_out, (cudaStream_t)stream);
}

int dmdqn_learn_stages(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                       const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, float* metrics_out,
                       void* workspace, size_t workspace_bytes, int32_t stages, void* stream) {
    return run_learn(dims, hp, replay, nets, draws, learn_mask, metrics_out, workspace, workspace_bytes, stages, nullptr, 0,
                     stream);
}

int dmdqn_learn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, float* metrics_out,
                void* workspace, size_t workspace_bytes, void* stream) {
    return run_learn(dims, hp, replay, nets, draws, learn_mask, metrics_out, workspace, workspace_bytes, kAllStages, nullptr,
                     0, stream);
}

int dmdqn_step_host(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                    const dmdqn_nets* nets, const dmdqn_step_block* blk, const void* host_block, void* device_block,
                    float* metrics_dev, float* metrics_host, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp && blk && host_block && device_block && metrics_dev && metrics_host, "step_host: NULL argument");
    rc = check_n_step(hp);            // before the copy and the push: a refused step changes nothing
    if (rc) return rc;
    rc = check_dueling(hp);
    if (rc) return rc;
    const size_t offs[6] = {blk->obs_off, blk->next_obs_off, blk->act_off, blk->rew_off, blk->done_off, blk->draws_off};
    for (size_t o : offs) DMDQN_CHECK_ARG(o % 16 == 0 && o < blk->bytes, "step_host: offset %zu is not a multiple of 16 inside the block", o);
    cudaStream_t s = (cudaStream_t)stream;
    char* d = static_cast<char*>(device_block);
    DMDQN_CUDA(cudaMemcpyAsync(d, host_block, blk->bytes, cudaMemcpyHostToDevice, s));
    rc = dmdqn_push(dims, replay, reinterpret_cast<const float*>(d + blk->obs_off), reinterpret_cast<const int32_t*>(d + blk->act_off),
                    reinterpret_cast<const double*>(d + blk->rew_off), reinterpret_cast<const float*>(d + blk->next_obs_off),
                    reinterpret_cast<const uint8_t*>(d + blk->done_off), blk->in_stride, nullptr, stream);
    if (rc) return rc;
    rc = dmdqn_learn(dims, hp, replay, nets, d + blk->draws_off, nullptr, metrics_dev, workspace, workspace_bytes, stream);
    if (rc) return rc;
    DMDQN_CUDA(cudaMemcpyAsync(metrics_host, metrics_dev, (size_t)dims->n_nets * DMDQN_METRICS_STRIDE * sizeof(float),
                               cudaMemcpyDeviceToHost, s));
    return DMDQN_OK;
}

int dmdqn_learn_grads(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                      const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t global_batch,
                      float* grads_out, float* metrics_out, void* workspace, size_t workspace_bytes, void* stream) {
    DMDQN_CHECK_ARG(grads_out != nullptr, "grads_out is NULL");
    return run_learn(dims, hp, replay, nets, draws, learn_mask, metrics_out, workspace, workspace_bytes, kAllStages,
                     grads_out, global_batch, stream);
}

int dmdqn_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const float* grads,
                     void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp && nets && nets->theta && nets->theta_tgt && nets->adam_m && nets->adam_v && grads,
                    "adam_apply: NULL argument");
    rc = check_dueling(hp);
    if (rc) return rc;
    return run_adam(*dims, *hp, {1, 1, hp->dueling == 1, 0}, *nets, grads, 0.0, nullptr, workspace, w, stream);
}

int dmdqn_clip_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const float* grads,
                          double global_clipnorm, float* norms_out, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp && nets && nets->theta && nets->theta_tgt && nets->adam_m && nets->adam_v && grads,
                    "clip_adam_apply: NULL argument");
    rc = check_dueling(hp);
    if (rc) return rc;
    DMDQN_CHECK_ARG(global_clipnorm > 0.0 && isfinite(global_clipnorm),
                    "global_clipnorm=%g must be a positive finite number", global_clipnorm);
    return run_adam(*dims, *hp, {1, 1, hp->dueling == 1, 0}, *nets, grads, global_clipnorm, norms_out, workspace, w, stream);
}

int dmdqn_allreduce_adam(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_peers* peers,
                         const float* my_loss_src, float* loss_out, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp && nets && nets->theta && nets->theta_tgt && nets->adam_m && nets->adam_v && peers && my_loss_src,
                    "allreduce_adam: NULL argument");
    rc = check_dueling(hp);
    if (rc) return rc;
    DMDQN_CHECK_ARG(dims->n_nets == 1, "allreduce_adam serves the shared network (n_nets == 1), got n_nets=%d", dims->n_nets);
    DMDQN_CHECK_ARG(peers->world >= 1 && peers->world <= DMDQN_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world,
                    "allreduce_adam: rank %d of world %d (at most %d peers)", peers->rank, peers->world, DMDQN_MAX_PEERS);
    DMDQN_CHECK_ARG(peers->epoch != 0, "allreduce_adam: epoch starts at 1 (the flag arrays are zero-initialised)");
    for (int p = 0; p < peers->world; ++p)
        DMDQN_CHECK_ARG(peers->grads[p] && peers->loss[p] && peers->flags[p], "allreduce_adam: NULL pointer for peer %d", p);
    return launch_peer_adam(*dims, *hp, *nets, *peers, my_loss_src, loss_out, (char*)workspace, w, (cudaStream_t)stream);
}

// CUDA IPC: the handle names a whole cudaMalloc allocation, so the offset of the pointer inside it travels along
// (a torch tensor is a slice of the caching allocator's block).  The driver entry point is looked up at run time
// (the library links cudart only).
int dmdqn_ipc_export(const void* dev_ptr, void* handle64, uint64_t* offset) {
    DMDQN_CHECK_ARG(dev_ptr && handle64 && offset, "ipc_export: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI carries the handle as 64 bytes");
    typedef int (*RangeFn)(unsigned long long*, size_t*, unsigned long long);
    static RangeFn range = nullptr;
    if (!range) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        DMDQN_CUDA(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q));
        if (q != cudaDriverEntryPointSuccess || !fn) {
            set_error("cuMemGetAddressRange is not available from this driver");
            return DMDQN_ERR_CUDA;
        }
        range = reinterpret_cast<RangeFn>(fn);
    }
    unsigned long long base = 0;
    size_t size = 0;
    const int drc = range(&base, &size, (unsigned long long)(uintptr_t)dev_ptr);
    if (drc != 0) {
        set_error("cuMemGetAddressRange failed with CUresult %d", drc);
        return DMDQN_ERR_CUDA;
    }
    cudaIpcMemHandle_t h;
    DMDQN_CUDA(cudaIpcGetMemHandle(&h, reinterpret_cast<void*>((uintptr_t)base)));
    memcpy(handle64, &h, sizeof(h));
    *offset = (uint64_t)((uintptr_t)dev_ptr - (uintptr_t)base);
    return DMDQN_OK;
}

int dmdqn_ipc_open(const void* handle64, uint64_t offset, void** dev_ptr) {
    DMDQN_CHECK_ARG(handle64 && dev_ptr, "ipc_open: NULL argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    void* base = nullptr;
    DMDQN_CUDA(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
    *dev_ptr = static_cast<char*>(base) + offset;
    return DMDQN_OK;
}

int dmdqn_ipc_close(void* dev_ptr, uint64_t offset) {
    DMDQN_CHECK_ARG(dev_ptr != nullptr, "ipc_close: NULL argument");
    DMDQN_CUDA(cudaIpcCloseMemHandle(static_cast<char*>(dev_ptr) - offset));
    return DMDQN_OK;
}

int dmdqn_debug(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_debug_views* out) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    char* ws = (char*)workspace;
    out->y = (const float*)(ws + w.y);
    out->q_all = (const float*)(ws + w.q_all);
    out->q_next = (const float*)(ws + w.q_next);
    out->tq_all = (const float*)(ws + w.tq_all);
    out->rows = (const int32_t*)(ws + w.rows);
    out->r_hat = (const float*)(ws + w.r_hat);
    out->active = (const int32_t*)(ws + w.active);
    out->tc_error = (const int32_t*)(ws + w.tc_error);
    out->dh1 = (const float*)(ws + w.dh1);
    out->dh2 = (const float*)(ws + w.dh2);
    out->relu2_bits = (const uint32_t*)(ws + w.mask2);
    out->is_w = (const float*)(ws + w.is_w);
    return DMDQN_OK;
}

int dmdqn_debug_nstep(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_nstep_views* out) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    out->next_rows = (const int32_t*)((char*)workspace + w.nrows);
    out->discount = (const float*)((char*)workspace + w.disc_b);
    return DMDQN_OK;
}

int dmdqn_debug_dueling(const dmdqn_dims* dims, void* workspace, size_t workspace_bytes, dmdqn_dueling_views* out) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    out->head = (const float*)((char*)workspace + w.head);
    return DMDQN_OK;
}

int dmdqn_noise_layout(const dmdqn_dims* dims, dmdqn_noise_record* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    copy_noise_rec(make_noise_rec(dims->obs_stride, dims->hidden), out);
    return DMDQN_OK;
}

static bool aligned16(const void* p) { return (uintptr_t)p % 16 == 0; }

// What every dmdqn_learn_grads_* call checks before it launches, besides the checks of its own arguments: the workspace,
// the learn arguments, the gradient block and global_batch.
static int check_learn_grads(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay, const dmdqn_nets* nets,
                             const void* draws, int32_t global_batch, const float* grads_out, void* workspace,
                             size_t workspace_bytes, Workspace* w) {
    int rc = check_workspace(dims, workspace, workspace_bytes, w);
    if (rc) return rc;
    if ((rc = check_learn_args(dims, hp, replay, nets, draws))) return rc;
    DMDQN_CHECK_ARG(grads_out && aligned16(grads_out), "grads_out is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(global_batch >= dims->batch, "global_batch=%d < batch=%d", global_batch, dims->batch);
    return DMDQN_OK;
}

// Every pointer of the noisy blocks, and the 16-byte alignment the float4 kernels need.
static int check_noisy(const dmdqn_nets* nets, const dmdqn_noisy* nz, bool adam) {
    DMDQN_CHECK_ARG(nets && nz && nets->theta && nets->theta_tgt && nets->learn_step, "noisy: NULL network pointer");
    DMDQN_CHECK_ARG(nz->sigma && nz->sigma_tgt && nz->eff && nz->eff_tgt && nz->noise && nz->key, "noisy: NULL noisy pointer");
    if (adam) DMDQN_CHECK_ARG(nets->adam_m && nets->adam_v && nz->sigma_m && nz->sigma_v, "noisy: NULL Adam moment pointer");
    const void* p[] = {nets->theta, nets->theta_tgt, nz->sigma, nz->sigma_tgt, nz->eff, nz->eff_tgt, nz->noise,
                       adam ? nz->sigma_m : nz->sigma, adam ? nz->sigma_v : nz->sigma};
    for (const void* q : p) DMDQN_CHECK_ARG((uintptr_t)q % 16 == 0, "noisy: pointer %p is not 16-byte aligned", q);
    return DMDQN_OK;
}

int dmdqn_noisy_fold(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                     void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp != nullptr, "noisy_fold: hp is NULL");
    if ((rc = check_dueling(hp))) return rc;
    if ((rc = check_noisy(nets, noisy, false))) return rc;
    return launch_noisy_fold(*dims, {1, 1, hp->dueling == 1, 0}, *nets, *noisy, (cudaStream_t)stream);
}

int dmdqn_learn_grads_noisy(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_replay* replay,
                            const dmdqn_nets* nets, const dmdqn_noisy* noisy, const void* draws, const uint8_t* learn_mask,
                            int32_t global_batch, float* grads_out, float* metrics_out, void* workspace,
                            size_t workspace_bytes, void* stream) {
    Workspace w;                      // everything run_learn checks, before the fold is launched
    int rc = check_learn_grads(dims, hp, replay, nets, draws, global_batch, grads_out, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_noisy(nets, noisy, true))) return rc;
    DMDQN_CHECK_ARG(hp->precision == DMDQN_PRECISION_FP32 || tc_supported(*dims),
                    "precision=%d (tcgen05) needs hidden=256 and obs_stride in {32,64,96}; got hidden=%d obs_stride=%d",
                    hp->precision, dims->hidden, dims->obs_stride);
    if ((rc = launch_noisy_fold(*dims, {1, 1, hp->dueling == 1, 0}, *nets, *noisy, (cudaStream_t)stream))) return rc;
    dmdqn_nets eff = *nets;
    eff.theta = noisy->eff;
    eff.theta_tgt = noisy->eff_tgt;
    return run_learn(dims, hp, replay, &eff, draws, learn_mask, metrics_out, workspace, workspace_bytes, kAllStages, grads_out,
                     global_batch, stream);
}

int dmdqn_noisy_adam_apply(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                           const float* grads, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    DMDQN_CHECK_ARG(hp && grads, "noisy_adam_apply: NULL argument");
    if ((rc = check_dueling(hp))) return rc;
    if ((rc = check_noisy(nets, noisy, true))) return rc;
    DMDQN_CHECK_ARG((uintptr_t)grads % 16 == 0, "noisy_adam_apply: grads is not 16-byte aligned");
    return launch_noisy_adam_apply(*dims, *hp, {1, 1, hp->dueling == 1, 0}, *nets, *noisy, grads, (char*)workspace, w,
                                   (cudaStream_t)stream);
}

int dmdqn_act_noisy(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t dueling,
                    const float* obs, int32_t obs_in_stride, const double* eps, const uint32_t* w_explore,
                    const uint32_t* w_action, int32_t* actions_out, float* q_out, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(dueling == 0 || dueling == 1, "dueling=%d must be 0 or 1", dueling);
    DMDQN_CHECK_ARG(nets && nets->theta && nets->learn_step && noisy && noisy->sigma && noisy->key, "act_noisy: NULL network pointer");
    DMDQN_CHECK_ARG((uintptr_t)nets->theta % 16 == 0 && (uintptr_t)noisy->sigma % 16 == 0,
                    "act_noisy: theta and sigma must be 16-byte aligned");
    DMDQN_CHECK_ARG(obs && eps && w_explore && w_action && actions_out, "act_noisy: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act(*dims, *nets, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out, dueling == 1,
                      (cudaStream_t)stream, noisy);
}

int dmdqn_sync_target_noisy(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t dueling,
                            const uint8_t* mask, double tau, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(dueling == 0 || dueling == 1, "dueling=%d must be 0 or 1", dueling);
    DMDQN_CHECK_ARG(nets && nets->theta && nets->theta_tgt && noisy && noisy->sigma && noisy->sigma_tgt,
                    "sync_target_noisy: NULL network pointer");
    return sync_noisy(*dims, {1, 1, dueling == 1, 0}, *nets, *noisy, mask, tau, stream);
}

// Distributional calls (include/dmdqn_b200.h dmdqn_dist): the atom count, the support and, where the call reads it, the
// scratch; every check runs before anything is launched.
static int check_atoms(int32_t n_atoms) {
    DMDQN_CHECK_ARG(n_atoms >= 2 && n_atoms <= DMDQN_DIST_MAX_ATOMS, "n_atoms=%d must be in [2, %d]", n_atoms,
                    DMDQN_DIST_MAX_ATOMS);
    return DMDQN_OK;
}

static int check_dist(const dmdqn_dims* dims, const dmdqn_dist* ds, bool scratch) {
    DMDQN_CHECK_ARG(ds != nullptr, "dist is NULL");
    if (int rc = check_atoms(ds->n_atoms)) return rc;
    DMDQN_CHECK_ARG(isfinite(ds->v_min) && isfinite(ds->v_max) && ds->v_min < ds->v_max,
                    "v_min=%g v_max=%g: the support needs finite v_min < v_max", ds->v_min, ds->v_max);
    if (scratch) {
        DMDQN_CHECK_ARG(ds->scratch && aligned16(ds->scratch), "dist: scratch is NULL or not 16-byte aligned");
        const size_t need = make_dist_scratch(*dims, dist_np(ds->n_atoms)).total;
        DMDQN_CHECK_ARG(ds->scratch_bytes >= need, "dist: scratch has %zu bytes, %zu needed", ds->scratch_bytes, need);
    }
    return DMDQN_OK;
}

// The hparams of the fp32-only kinds: `tag` names the call family, `kind` the networks; `dueling` is the hp->dueling the
// block needs (1: it carries a value stream), `note` trails the refusal of a dueling head where none is supported.
static int check_kind_hp(const dmdqn_hparams* hp, const char* tag, const char* kind, int32_t dueling, const char* note = "") {
    DMDQN_CHECK_ARG(hp != nullptr, "%s: hp is NULL", tag);
    DMDQN_CHECK_ARG(hp->precision == DMDQN_PRECISION_FP32, "precision=%d: %s networks run the fp32 (FFMA) path only",
                    hp->precision, kind);
    if (dueling)
        DMDQN_CHECK_ARG(hp->dueling == 1, "dueling=%d: %s blocks carry the value stream, so hp->dueling must be 1", hp->dueling,
                        kind);
    else
        DMDQN_CHECK_ARG(hp->dueling == 0, "dueling=%d: dueling heads are not supported with %s networks%s", hp->dueling, kind,
                        note);
    return DMDQN_OK;
}
static int check_dist_hp(const dmdqn_hparams* hp) {
    return check_kind_hp(hp, "dist", "distributional", 0, " (dueling noisy C51 heads: the dmdqn_*_rainbow calls)");
}


static int check_dist_nets(const dmdqn_nets* nets, bool adam) {
    DMDQN_CHECK_ARG(nets && nets->theta && nets->theta_tgt, "dist: NULL network pointer");
    if (adam) DMDQN_CHECK_ARG(nets->adam_m && nets->adam_v && nets->learn_step, "dist: NULL Adam pointer");
    const void* p[] = {nets->theta, nets->theta_tgt, adam ? nets->adam_m : nets->theta, adam ? nets->adam_v : nets->theta};
    for (const void* q : p) DMDQN_CHECK_ARG(aligned16(q), "dist: pointer %p is not 16-byte aligned", q);
    return DMDQN_OK;
}

int dmdqn_param_layout_dist(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_layout* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    copy_trunk(make_layout(dims->obs_stride, dims->hidden, atom_shape(n_atoms, false)), out);
    return DMDQN_OK;
}

int dmdqn_dist_scratch_bytes(const dmdqn_dims* dims, int32_t n_atoms, size_t* out_bytes) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    DMDQN_CHECK_ARG(out_bytes != nullptr, "out_bytes is NULL");
    *out_bytes = make_dist_scratch(*dims, dist_np(n_atoms)).total;
    return DMDQN_OK;
}

int dmdqn_learn_grads_dist(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_dist* dist, const dmdqn_replay* replay,
                           const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t global_batch,
                           float* grads_out, float* metrics_out, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_learn_grads(dims, hp, replay, nets, draws, global_batch, grads_out, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_dist_hp(hp))) return rc;
    if ((rc = check_dist(dims, dist, true))) return rc;
    if ((rc = check_dist_nets(nets, true))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = launch_sample(*dims, *hp, *replay, *nets, draws, learn_mask, 1, (char*)workspace, w, s))) return rc;
    return launch_learn_dist(*dims, *hp, *replay, *nets, *dist, metrics_out, (char*)workspace, w, grads_out, global_batch, s);
}

int dmdqn_adam_apply_dist(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, int32_t n_atoms,
                          const float* grads, double global_clipnorm, float* norms_out, void* workspace, size_t workspace_bytes,
                          void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_dist_hp(hp))) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    if ((rc = check_dist_nets(nets, true))) return rc;
    DMDQN_CHECK_ARG(grads && aligned16(grads), "adam_apply_dist: grads is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(global_clipnorm >= 0.0 && isfinite(global_clipnorm),
                    "global_clipnorm=%g must be 0 (no clipping) or a positive finite number", global_clipnorm);
    return run_adam(*dims, *hp, atom_shape(n_atoms, false), *nets, grads, global_clipnorm, norms_out, workspace, w, stream);
}

int dmdqn_act_dist(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_dist* dist, const float* obs,
                   int32_t obs_in_stride, const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
                   int32_t* actions_out, float* q_out, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_dist(dims, dist, false))) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && aligned16(nets->theta), "act_dist: theta is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(obs && eps && w_explore && w_action && actions_out, "act_dist: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act_dist(*dims, *nets, *dist, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out,
                           (cudaStream_t)stream);
}

int dmdqn_sync_target_dist(const dmdqn_dims* dims, const dmdqn_nets* nets, int32_t n_atoms, const uint8_t* mask, double tau,
                           void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    if ((rc = check_dist_nets(nets, false))) return rc;
    return launch_sync_target(*dims, make_layout(dims->obs_stride, dims->hidden, atom_shape(n_atoms, false)).stride, nets->theta,
                              nets->theta_tgt, mask, tau, (cudaStream_t)stream);
}

int dmdqn_debug_dist(const dmdqn_dims* dims, const dmdqn_dist* dist, dmdqn_dist_views* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_dist(dims, dist, true))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const DistArgs D = make_dist_args(*dims, *dist);
    out->target_dist = D.m;
    out->h2 = D.h2;
    out->dlogits = D.dx;
    return DMDQN_OK;
}

// Quantile calls (include/dmdqn_b200.h dmdqn_quantile): the quantile count, kappa and, where the call reads it, the scratch;
// the hparams and network checks are those of the distributional calls.
static int check_quantile(const dmdqn_dims* dims, const dmdqn_quantile* qs, bool scratch) {
    DMDQN_CHECK_ARG(qs != nullptr, "quantile is NULL");
    DMDQN_CHECK_ARG(qs->n_quantiles >= 2 && qs->n_quantiles <= DMDQN_DIST_MAX_ATOMS, "n_quantiles=%d must be in [2, %d]",
                    qs->n_quantiles, DMDQN_DIST_MAX_ATOMS);
    DMDQN_CHECK_ARG(isfinite(qs->kappa) && qs->kappa >= 0.0, "kappa=%g must be finite and >= 0", qs->kappa);
    if (scratch) {
        DMDQN_CHECK_ARG(qs->scratch && aligned16(qs->scratch), "quantile: scratch is NULL or not 16-byte aligned");
        const size_t need = make_dist_scratch(*dims, dist_np(qs->n_quantiles)).total;
        DMDQN_CHECK_ARG(qs->scratch_bytes >= need, "quantile: scratch has %zu bytes, %zu needed", qs->scratch_bytes, need);
    }
    return DMDQN_OK;
}

int dmdqn_learn_grads_quantile(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_quantile* quantile,
                               const dmdqn_replay* replay, const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask,
                               int32_t global_batch, float* grads_out, float* metrics_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_learn_grads(dims, hp, replay, nets, draws, global_batch, grads_out, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_dist_hp(hp))) return rc;
    if ((rc = check_quantile(dims, quantile, true))) return rc;
    if ((rc = check_dist_nets(nets, true))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = launch_sample(*dims, *hp, *replay, *nets, draws, learn_mask, 1, (char*)workspace, w, s))) return rc;
    return launch_learn_quantile(*dims, *hp, *replay, *nets, *quantile, metrics_out, (char*)workspace, w, grads_out,
                                 global_batch, s);
}

int dmdqn_act_quantile(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_quantile* quantile, const float* obs,
                       int32_t obs_in_stride, const double* eps, const uint32_t* w_explore, const uint32_t* w_action,
                       int32_t* actions_out, float* q_out, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_quantile(dims, quantile, false))) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && aligned16(nets->theta), "act_quantile: theta is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(obs && eps && w_explore && w_action && actions_out, "act_quantile: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act_quantile(*dims, *nets, *quantile, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out,
                               (cudaStream_t)stream);
}

int dmdqn_debug_quantile(const dmdqn_dims* dims, const dmdqn_quantile* quantile, dmdqn_dist_views* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_quantile(dims, quantile, true))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const QuantArgs Q = make_quantile_args(*dims, *quantile);
    out->target_dist = Q.m;
    out->h2 = Q.h2;
    out->dlogits = Q.dx;
    return DMDQN_OK;
}

// IQN calls (include/dmdqn_b200.h dmdqn_iqn): the counts, n_cos, kappa, row_base and, where the call reads them, the key and
// the scratch; every check runs before anything is launched.
static int check_n_cos(int32_t n_cos) {
    DMDQN_CHECK_ARG(n_cos >= 4 && n_cos <= DMDQN_IQN_MAX_COS && n_cos % 4 == 0, "n_cos=%d must be a multiple of 4 in [4, %d]",
                    n_cos, DMDQN_IQN_MAX_COS);
    return DMDQN_OK;
}

static int check_iqn(const dmdqn_dims* dims, const dmdqn_iqn* q, bool learn) {
    DMDQN_CHECK_ARG(q != nullptr, "iqn is NULL");
    const int32_t counts[3] = {q->n_tau, q->n_tau_prime, q->n_policy};
    const char* names[3] = {"n_tau", "n_tau_prime", "n_policy"};
    for (int i = 0; i < 3; ++i)
        DMDQN_CHECK_ARG(counts[i] >= 1 && counts[i] <= DMDQN_IQN_MAX_TAU, "%s=%d must be in [1, %d]", names[i], counts[i],
                        DMDQN_IQN_MAX_TAU);
    if (int rc = check_n_cos(q->n_cos)) return rc;
    DMDQN_CHECK_ARG(isfinite(q->kappa) && q->kappa >= 0.0, "kappa=%g must be finite and >= 0", q->kappa);
    DMDQN_CHECK_ARG(q->row_base >= 0, "row_base=%lld must be >= 0", (long long)q->row_base);
    if (learn) {
        DMDQN_CHECK_ARG(q->key != nullptr, "iqn: key is NULL");
        DMDQN_CHECK_ARG(q->scratch && aligned16(q->scratch), "iqn: scratch is NULL or not 16-byte aligned");
        const size_t need = make_iqn_scratch(*dims, q->n_tau, q->n_tau_prime, q->n_cos).total;
        DMDQN_CHECK_ARG(q->scratch_bytes >= need, "iqn: scratch has %zu bytes, %zu needed", q->scratch_bytes, need);
    }
    return DMDQN_OK;
}

static int check_iqn_hp(const dmdqn_hparams* hp) { return check_kind_hp(hp, "iqn", "IQN", 0); }

int dmdqn_param_layout_iqn(const dmdqn_dims* dims, int32_t n_cos, dmdqn_iqn_layout* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_n_cos(n_cos))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const Layout l = make_layout(dims->obs_stride, dims->hidden, {1, 1, false, n_cos});
    copy_trunk(l, out);
    out->wphi = l.wphi; out->bphi = l.bphi; out->end = l.end;
    return DMDQN_OK;
}

int dmdqn_iqn_scratch_bytes(const dmdqn_dims* dims, const dmdqn_iqn* iqn, size_t* out_bytes) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_iqn(dims, iqn, false))) return rc;
    DMDQN_CHECK_ARG(out_bytes != nullptr, "out_bytes is NULL");
    *out_bytes = make_iqn_scratch(*dims, iqn->n_tau, iqn->n_tau_prime, iqn->n_cos).total;
    return DMDQN_OK;
}

int dmdqn_learn_grads_iqn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_iqn* iqn, const dmdqn_replay* replay,
                          const dmdqn_nets* nets, const void* draws, const uint8_t* learn_mask, int32_t global_batch,
                          float* grads_out, float* metrics_out, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_learn_grads(dims, hp, replay, nets, draws, global_batch, grads_out, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_iqn_hp(hp))) return rc;
    if ((rc = check_iqn(dims, iqn, true))) return rc;
    if ((rc = check_dist_nets(nets, true))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = launch_sample(*dims, *hp, *replay, *nets, draws, learn_mask, 1, (char*)workspace, w, s))) return rc;
    return launch_learn_iqn(*dims, *hp, *replay, *nets, *iqn, metrics_out, (char*)workspace, w, grads_out, global_batch, s);
}

int dmdqn_adam_apply_iqn(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, int32_t n_cos,
                         const float* grads, double global_clipnorm, float* norms_out, void* workspace, size_t workspace_bytes,
                         void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_iqn_hp(hp))) return rc;
    if ((rc = check_n_cos(n_cos))) return rc;
    if ((rc = check_dist_nets(nets, true))) return rc;
    DMDQN_CHECK_ARG(grads && aligned16(grads), "adam_apply_iqn: grads is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(global_clipnorm >= 0.0 && isfinite(global_clipnorm),
                    "global_clipnorm=%g must be 0 (no clipping) or a positive finite number", global_clipnorm);
    return run_adam(*dims, *hp, {1, 1, false, n_cos}, *nets, grads, global_clipnorm, norms_out, workspace, w, stream);
}

int dmdqn_act_iqn(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_iqn* iqn, const float* obs, int32_t obs_in_stride,
                  const double* eps, const uint32_t* w_explore, const uint32_t* w_action, int32_t* actions_out, float* q_out,
                  void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_iqn(dims, iqn, false))) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && aligned16(nets->theta), "act_iqn: theta is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(obs && eps && w_explore && w_action && actions_out, "act_iqn: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act_iqn(*dims, *nets, *iqn, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out,
                          (cudaStream_t)stream);
}

int dmdqn_sync_target_iqn(const dmdqn_dims* dims, const dmdqn_nets* nets, int32_t n_cos, const uint8_t* mask, double tau,
                          void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_n_cos(n_cos))) return rc;
    if ((rc = check_dist_nets(nets, false))) return rc;
    return launch_sync_target(*dims, make_layout(dims->obs_stride, dims->hidden, {1, 1, false, n_cos}).stride, nets->theta,
                              nets->theta_tgt, mask, tau, (cudaStream_t)stream);
}

int dmdqn_debug_iqn(const dmdqn_dims* dims, const dmdqn_iqn* iqn, dmdqn_iqn_views* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_iqn(dims, iqn, false))) return rc;
    DMDQN_CHECK_ARG(iqn->scratch && aligned16(iqn->scratch), "iqn: scratch is NULL or not 16-byte aligned");
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const IqnArgs Q = make_iqn_args(*dims, *iqn);
    out->tau = Q.tau; out->tau_prime = Q.tau_p; out->target = Q.t; out->theta = Q.theta; out->grad = Q.grad;
    out->dh2 = Q.h2; out->dphi = Q.phi;
    return DMDQN_OK;
}

// Rainbow calls (include/dmdqn_b200.h dmdqn_rainbow_layout): dmdqn_dist's atom and support checks, the Rainbow scratch,
// dueling == 1 where hparams are taken, and dmdqn_noisy's pointer checks; every check runs before anything is launched.
static int check_rainbow(const dmdqn_dims* dims, const dmdqn_dist* ds, bool scratch) {
    if (int rc = check_dist(dims, ds, false)) return rc;
    if (scratch) {
        DMDQN_CHECK_ARG(ds->scratch && aligned16(ds->scratch), "rainbow: scratch is NULL or not 16-byte aligned");
        const size_t need = make_rainbow_scratch(*dims, dist_np(ds->n_atoms)).total;
        DMDQN_CHECK_ARG(ds->scratch_bytes >= need, "rainbow: scratch has %zu bytes, %zu needed", ds->scratch_bytes, need);
    }
    return DMDQN_OK;
}

static int check_rainbow_hp(const dmdqn_hparams* hp) { return check_kind_hp(hp, "rainbow", "Rainbow", 1); }

int dmdqn_param_layout_rainbow(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_rainbow_layout* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const Layout l = make_layout(dims->obs_stride, dims->hidden, atom_shape(n_atoms, true));
    copy_trunk(l, out);
    out->wv = l.wv; out->bv = l.bv; out->end = l.end;
    return DMDQN_OK;
}

int dmdqn_noise_layout_rainbow(const dmdqn_dims* dims, int32_t n_atoms, dmdqn_noise_record* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    copy_noise_rec(make_noise_rec(dims->obs_stride, dims->hidden, atom_shape(n_atoms, true)), out);
    return DMDQN_OK;
}

int dmdqn_rainbow_scratch_bytes(const dmdqn_dims* dims, int32_t n_atoms, size_t* out_bytes) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    DMDQN_CHECK_ARG(out_bytes != nullptr, "out_bytes is NULL");
    *out_bytes = make_rainbow_scratch(*dims, dist_np(n_atoms)).total;
    return DMDQN_OK;
}

int dmdqn_rainbow_fold(const dmdqn_dims* dims, const dmdqn_dist* dist, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                       void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_rainbow(dims, dist, true))) return rc;
    if ((rc = check_noisy(nets, noisy, false))) return rc;
    return launch_rainbow_fold(*dims, *dist, *nets, *noisy, (cudaStream_t)stream);
}

int dmdqn_learn_grads_rainbow(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_dist* dist,
                              const dmdqn_replay* replay, const dmdqn_nets* nets, const dmdqn_noisy* noisy, const void* draws,
                              const uint8_t* learn_mask, int32_t global_batch, float* grads_out, float* metrics_out,
                              void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_learn_grads(dims, hp, replay, nets, draws, global_batch, grads_out, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_rainbow_hp(hp))) return rc;
    if ((rc = check_rainbow(dims, dist, true))) return rc;
    if ((rc = check_noisy(nets, noisy, true))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = launch_rainbow_fold(*dims, *dist, *nets, *noisy, s))) return rc;
    dmdqn_nets eff = *nets;
    eff.theta = noisy->eff;
    eff.theta_tgt = noisy->eff_tgt;
    if ((rc = launch_sample(*dims, *hp, *replay, eff, draws, learn_mask, 1, (char*)workspace, w, s))) return rc;
    return launch_learn_rainbow(*dims, *hp, *replay, eff, *dist, metrics_out, (char*)workspace, w, grads_out, global_batch, s);
}

int dmdqn_adam_apply_rainbow(const dmdqn_dims* dims, const dmdqn_hparams* hp, const dmdqn_nets* nets, const dmdqn_noisy* noisy,
                             int32_t n_atoms, const float* grads, void* workspace, size_t workspace_bytes, void* stream) {
    Workspace w;
    int rc = check_workspace(dims, workspace, workspace_bytes, &w);
    if (rc) return rc;
    if ((rc = check_rainbow_hp(hp))) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    if ((rc = check_noisy(nets, noisy, true))) return rc;
    DMDQN_CHECK_ARG(grads && aligned16(grads), "adam_apply_rainbow: grads is NULL or not 16-byte aligned");
    return launch_noisy_adam_apply(*dims, *hp, atom_shape(n_atoms, true), *nets, *noisy, grads, (char*)workspace, w,
                                   (cudaStream_t)stream);
}

int dmdqn_act_rainbow(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, const dmdqn_dist* dist,
                      const float* obs, int32_t obs_in_stride, const double* eps, const uint32_t* w_explore,
                      const uint32_t* w_action, int32_t* actions_out, float* q_out, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_rainbow(dims, dist, false))) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && aligned16(nets->theta), "act_rainbow: theta is NULL or not 16-byte aligned");
    if (noisy)
        DMDQN_CHECK_ARG(noisy->sigma && aligned16(noisy->sigma) && noisy->key && nets->learn_step,
                        "act_rainbow: sigma, key or learn_step is NULL, or sigma is not 16-byte aligned");
    DMDQN_CHECK_ARG(obs && eps && w_explore && w_action && actions_out, "act_rainbow: NULL argument");
    DMDQN_CHECK_ARG(obs_in_stride >= dims->obs_dim, "obs_in_stride=%d < obs_dim=%d", obs_in_stride, dims->obs_dim);
    return launch_act_rainbow(*dims, *nets, noisy, *dist, obs, obs_in_stride, eps, w_explore, w_action, actions_out, q_out,
                              (cudaStream_t)stream);
}

int dmdqn_sync_target_rainbow(const dmdqn_dims* dims, const dmdqn_nets* nets, const dmdqn_noisy* noisy, int32_t n_atoms,
                              const uint8_t* mask, double tau, void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_atoms(n_atoms))) return rc;
    if ((rc = check_noisy(nets, noisy, false))) return rc;
    return sync_noisy(*dims, atom_shape(n_atoms, true), *nets, *noisy, mask, tau, stream);
}

int dmdqn_debug_rainbow(const dmdqn_dims* dims, const dmdqn_dist* dist, dmdqn_rainbow_views* out) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    if ((rc = check_rainbow(dims, dist, true))) return rc;
    DMDQN_CHECK_ARG(out != nullptr, "out is NULL");
    const DistArgs D = make_dist_args(*dims, *dist);
    out->target_dist = D.m;
    out->h2 = D.h2;
    out->dlogits = D.dx;
    out->head = reinterpret_cast<const float*>(static_cast<const char*>(dist->scratch) + make_rainbow_scratch(*dims, D.np).head);
    return DMDQN_OK;
}

static int run_sync_target(const dmdqn_dims* dims, const dmdqn_nets* nets, const uint8_t* mask, double tau, bool dueling,
                           void* stream) {
    int rc = validate_dims(dims);
    if (rc) return rc;
    DMDQN_CHECK_ARG(nets && nets->theta && nets->theta_tgt, "sync_target: NULL network pointer");
    return launch_sync_target(*dims, make_layout(dims->obs_stride, dims->hidden, {1, 1, dueling, 0}).stride, nets->theta,
                              nets->theta_tgt, mask, tau, (cudaStream_t)stream);
}

int dmdqn_sync_target(const dmdqn_dims* dims, const dmdqn_nets* nets, const uint8_t* mask, double tau,
                      void* stream) {
    return run_sync_target(dims, nets, mask, tau, false, stream);
}

int dmdqn_sync_target_dueling(const dmdqn_dims* dims, const dmdqn_nets* nets, const uint8_t* mask, double tau,
                              void* stream) {
    return run_sync_target(dims, nets, mask, tau, true, stream);
}

}  // extern "C"
