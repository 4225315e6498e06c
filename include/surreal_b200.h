/* libsurreal_b200 -- C-ABI of the B200-native actor -> replay -> learner hot path.
 *
 * The reference (SurrealAI/surreal) is pure Python and has NO FFI / operator registry: its plugin
 * surface is three Python base classes (Agent / Replay / Learner, SURVEY.md §8b).  This header is
 * therefore the boundary a maintainer would bind from those classes (ctypes stub in
 * INTEGRATION.md); every entry point cites the reference code whose arithmetic it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _h; fp32, row-major, contiguous
 *     unless a leading dimension is given; `stream` is a cudaStream_t passed as void*.
 *   - every call is asynchronous on `stream`, allocates nothing, and returns SB200_OK (0) or a
 *     negative sb200 status; no exceptions cross the ABI.  Workspaces are caller-owned.
 *   - weights use the KERNEL LAYOUT: W[l] is [in_l][ldw_l] (ldw = out rounded up to 4), i.e. the
 *     transpose of torch.nn.Linear.weight, zero in the padding columns; b[l] is [ldw_l].
 *   - there is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef SURREAL_B200_H
#define SURREAL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB200_OK 0
#define SB200_ERR_ARG (-1)
#define SB200_ERR_CUDA (-2)
#define SB200_ERR_UNSUPPORTED (-3)

#define SB200_ACT_NONE 0
#define SB200_ACT_RELU 1
#define SB200_ACT_TANH 2
#define SB200_MAX_LAYERS 4

int sb200_version(void);
/* One-time per-process setup on the current device (kernel attributes); fails on non-sm_100 devices.
 * Must run before any compute entry (and before CUDA-graph capture). */
int sb200_init(void);
const char* sb200_status_string(int status);
/* SM count / compute capability of the current device (fails without a GPU). */
int sb200_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Number of CUDA kernels this library has launched so far (optionally reset) -- bench.py's gpu_launches. */
uint64_t sb200_launch_counter(int reset);
/* Account for kernels submitted through a replayed CUDA graph (counted once at capture time). */
void sb200_launch_counter_add(uint64_t kernels);

/* ---------------------------------------------------------------------------------------------
 * Networks.  One descriptor covers PPO_ActorNetwork / PPO_CriticNetwork
 * (surreal/model/model_builders/builders.py:86-175), ActorNetworkX / CriticNetworkX (:35-84).
 * `aux_layer` >= 0 concatenates `aux` columns to the input of that layer (the DDPG critic's
 * cat(h, action), builders.py:80-83). */
typedef struct {
    int n_layers;                       /* 1..SB200_MAX_LAYERS */
    int dims[SB200_MAX_LAYERS + 1];     /* dims[0] = input width (without aux), dims[l+1] = out of layer l */
    int act[SB200_MAX_LAYERS];          /* SB200_ACT_* applied after layer l */
    const float* W[SB200_MAX_LAYERS];   /* [in_l(+aux)][ldw_l] */
    const float* b[SB200_MAX_LAYERS];   /* [ldw_l] */
    int ldw[SB200_MAX_LAYERS];
    int aux_layer;                      /* -1: none */
    int aux_dim;
} sb200_mlp;

/* ZFilter (surreal/model/z_filter.py:59-79): stats = running_sum[D] | running_sumsq[D] | count[1]. */
typedef struct {
    const float* stats;                 /* NULL: no filter */
    float eps;                          /* 1e-5 in the reference */
} sb200_zfilter;

/* Input rows of a forward pass.  Either a plain matrix (x, ldx, rows) or, when win_n > 0, the
 * virtual concatenation cat([obs, obs_next], dim=1).view(-1, D) of ppo.py:376-383 WITHOUT copying:
 * row r -> (b, k) = (r / (win_n+1), r % (win_n+1)); k < win_n ? x[(b*win_n+k)*ldx] : x_next[b*ldx]. */
typedef struct {
    const float* x;
    const float* x_next;                /* only when win_n > 0 */
    int64_t ldx;
    int64_t rows;                       /* total rows ( = B*(win_n+1) when win_n > 0 ) */
    int win_n;
    const float* aux;                   /* [rows][aux_ld] or NULL */
    int64_t aux_ld;
    float* save_x;                      /* optional: receives the z-filtered input rows [rows][ld_save_x] */
    int64_t ld_save_x;
} sb200_rows;

/* Fused forward of a whole MLP on row tiles (z-filter -> Linear/act x n_layers): activations stay in
 * shared memory; `save[l]` (may be NULL) receives layer l's post-activation output [rows][ld_save[l]]
 * (needed by the backward pass); save[n_layers-1] is the network output.
 * Replaces: ppo_net.py:253-315 (forward_actor / forward_critic), builders.py:114-132,160-175,
 * ddpg_net.py:63-91. */
int sb200_mlp_forward_f32(const sb200_mlp* net, const sb200_zfilter* zf, const sb200_rows* in,
                          float* const* save, const int64_t* ld_save, void* stream);
/* Same, with the kernel family chosen by the caller: variant 0 = default dispatch, 1 = tensor-core 3xTF32 tiles of
 * 32 rows, 2 = fp32 FFMA tiles of 32 rows (both <= 128 registers per thread, 2 CTAs/SM).  Variant 1 is what large
 * batches get by default (631 us on the 132 096-row critic pass).  Launching 1 and 2 on two streams over the two
 * halves of a batch -- tensor pipe and FMA pipe at once -- was measured SLOWER (700-760 us): both kernels are bound
 * by instruction issue, not by their math pipes; it stays available as an experiment (SB200_DUAL_CRITIC=1). */
int sb200_mlp_forward_variant_f32(const sb200_mlp* net, const sb200_zfilter* zf, const sb200_rows* in,
                                  float* const* save, const int64_t* ld_save, int variant, void* stream);
/* Small-batch inference on PRE-PACKED weights (the actors' per-step policy forward, ppo_agent.py:138-141 /
 * ddpg_agent.py:170-176): pack once per parameter version, then every step's forward reads the weights in
 * mma-fragment order and a 4-CTA cluster shares each 32-row tile (each CTA keeps a quarter of the weights resident in
 * shared memory and exchanges layer outputs through distributed shared memory).
 *   pack_floats: size of `packed` in floats (0: this architecture is not supported -- use sb200_mlp_forward_f32;
 *     supported = every layer but the last wider than 32 outputs).
 *   pack_tf32: (re)builds `packed` from net->W.  Must be re-run after ANY change of the parameters.
 *   forward_packed: out[rows][ld_out] = network output; same numerics class as forward mode 1. */
size_t sb200_mlp_pack_floats(const sb200_mlp* net);
int sb200_mlp_pack_tf32(const sb200_mlp* net, float* packed, void* stream);
int sb200_mlp_forward_packed_f32(const sb200_mlp* net, const float* packed, const sb200_zfilter* zf,
                                 const sb200_rows* in, float* out, int64_t ld_out, void* stream);
/* Blackwell-native large-batch forward (csrc/mlp_fwd_tc5.cu): tcgen05.mma kind::tf32 tiles of 128 rows with the
 * accumulators in tensor memory, weights streamed by the TMA engine (cp.async.bulk), 3xTF32 split for fp32-level
 * accuracy, both hidden layers and the narrow head fused in one persistent kernel (one CTA per SM).  The critic pass of
 * PPOLearner._gae_and_return (ppo.py:376-387: B*(n+1) rows through D-256-256-1) is its customer.
 *   supported: 3 layers, ReLU-ReLU-any, dims[0] a multiple of 32 up to 256, dims[1] multiple of 32 and dims[2] multiple of 64 (both
 *     <= 256), dims[3] <= 8, no aux input, rows >= 128.  Returns 1 / 0.
 *   workspace_bytes: caller-owned scratch for the per-call weight images (hi / lo planes in operand layout); 0 when
 *     unsupported.  One workspace must not be shared by calls that may run concurrently.
 *   forward: out[rows][ld_out] = network output (only the last layer is written: no saved activations, no save_x).
 *     SB200_ERR_UNSUPPORTED for other shapes -- callers then use sb200_mlp_forward_f32. */
int sb200_mlp_tc5_supported(const sb200_mlp* net, int64_t rows);
size_t sb200_mlp_tc5_workspace_bytes(const sb200_mlp* net);
int sb200_mlp_forward_tc5_f32(const sb200_mlp* net, const sb200_zfilter* zf, const sb200_rows* in, float* out,
                              int64_t ld_out, void* workspace, void* stream);
/* ---------------------------------------------------------------------------------------------
 * CNN stem of the pixel path (CNNStemNetwork, builders.py:8-33; used by PPOModel / DDPGModel with pixel input,
 * ppo_net.py:136-140,268-273,368-375): Conv2d(16, k8, s4)+ReLU -> Conv2d(32, k4, s2)+ReLU -> Flatten -> Linear+ReLU.
 * The two convolutions (csrc/stem.cu); the Linear layer is an ordinary sb200_mlp layer.
 *   frames [rows][C][H][W] (uint8 scaled by in_scale = 1/255, or float); outputs [rows][COUT][HO][WO] (torch order);
 *   Wk: kernel layout [(c*KS + ky)*KS + kx][COUT] = transpose of torch's [COUT][C][KS][KS]; bias [COUT].
 *   layer 1 = Conv2d(16, k8, s4), layer 2 = Conv2d(32, k4, s2) (the reference's fixed stem).
 *   forward: y = relu(conv(x * in_scale) + bias).
 *   backward_dw: partial gradients of `frames` frames w.r.t. Wk / bias, written into `splits` slabs at
 *     slab_w + s*slab_stride / slab_b + s*slab_stride (reduce with sb200_grad_reduce_norm_f32); dy = gradient w.r.t. the
 *     PRE-activation output.
 *   backward_dx (layer 2 only): dx = relu'(act) * conv_transpose(dy), act = layer 1's output (may be NULL: no mask). */
int sb200_conv_forward_f32(int layer, const void* x, int in_u8, int64_t frames, int CIN, int H, int W, const float* Wk,
                           const float* bias, double in_scale, float* y, void* stream);
int sb200_conv_backward_dw_f32(int layer, const void* x, int in_u8, const float* dy, int64_t frames, int CIN, int H, int W,
                               double in_scale, float* slab_w, float* slab_b, int64_t slab_stride, int splits, void* stream);
int sb200_conv_backward_dx_f32(int layer, const float* dy, const float* Wk, const float* act, int64_t frames, int CIN, int H,
                               int W, float* dx, void* stream);
/* Conv layer 1 forward / weight gradient on uint8 frames that sit `row_bytes` apart (>= CIN*H*W) instead of back to back:
 * the stem reads frames in place from wider records (the mixed pixel + low-dim observation rows).  With row_bytes = CIN*H*W
 * these are exactly sb200_conv_forward_f32 / sb200_conv_backward_dw_f32 for layer 1 with in_u8 = 1. */
int sb200_conv1_forward_u8_strided(const void* x, int64_t row_bytes, int64_t frames, int CIN, int H, int W, const float* Wk,
                                   const float* bias, double in_scale, float* y, void* stream);
int sb200_conv1_backward_dw_u8_strided(const void* x, int64_t row_bytes, const float* dy, int64_t frames, int CIN, int H, int W,
                                       double in_scale, float* slab_w, float* slab_b, int64_t slab_stride, int splits,
                                       void* stream);

/* One step of the device-resident synthetic PIXEL env (SURVEY §8d cfg 4: uint8 frames of uniform random bytes, reward
 * -mean(a^2) + 0.1 N(0,1), done at the episode cap): state = the frames the actors observe next, obs_next = true successors. */
int sb200_synth_pixel_env_step_u8(void* state, const float* action, int N, int64_t frame_bytes, int A, int max_steps,
                                  int* ep_step, uint64_t seed, const uint64_t* step_counter, void* obs_next, float* reward,
                                  float* done, void* stream);

/* One step of the device-resident synthetic MIXED env: packed observation rows [N][row_words] = frame (frame_words 32-bit
 * words of uint8 pixels, as synth_pixel_env) | D low-dim floats (dynamics, reward and done as synth_env) | zero padding.
 * state = the rows the actors observe next, obs_next = true successors (same layout).  Ws / Wa in synth_env's layout. */
int sb200_synth_mixed_env_step_f32(float* state, const float* action, const float* Ws, const float* Wa, int N, int D, int A,
                                   int frame_words, int64_t row_words, int max_steps, int* ep_step, uint64_t seed,
                                   const uint64_t* step_counter, float* obs_next, float* reward, float* done, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One-shot all-reduce over NVLink peer memory (csrc/peer_allreduce.cu) for the small exchanges of the data-parallel
 * learner (SURVEY §8e; the reference has no collective at all): every rank maps every other rank's "symmetric" buffer
 * (cudaMalloc + CUDA IPC), one kernel per all-reduce publishes its slice, waits for the peers' flags and sums the slots
 * in rank order (bit-identical result on all ranks).
 *   par_alloc / par_open / par_close: allocate + export (64-byte IPC handle) / map a peer's buffer / release.
 *   par_allreduce_f32: out = scale * sum over ranks of x (n <= max_floats); with opt_workspace != NULL it also does
 *     the gradient-norm / step bookkeeping of sb200_grad_reduce_norm_f32 on the result.  EVERY rank must issue the
 *     same sequence of calls on one sb200_par (use separate ones for streams that run concurrently).
 *   par_allreduce_f64: the same for a few float64 scalars. */
typedef struct {
    void* peers[8];                     /* device pointers of every rank's symmetric buffer, valid in THIS process */
    int world;
    int rank;
    int64_t max_floats;                 /* capacity of one slot */
} sb200_par;
size_t sb200_par_buffer_bytes(int64_t max_floats);
int sb200_par_alloc(int64_t max_floats, void** ptr_out, void* handle_out);
int sb200_par_open(const void* handle, void** ptr_out);
int sb200_par_close(void* ptr, int own);
int sb200_par_allreduce_f32(const sb200_par* ctx, const float* x, float* out, int64_t n, double scale, int bump_step,
                            void* opt_workspace, const int* stop_flag, void* stream);
int sb200_par_allreduce_f64(const sb200_par* ctx, const double* x, double* out, int n, double scale, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Persistent learner kernel (csrc/epoch2.cu): ALL minibatch epochs of BOTH optimisers of PPOLearner._optimize
 * (surreal/learner/ppo.py:194-353 losses + updates, 541-557 epoch loops + KL early stop) in ONE launch of one CTA per SM --
 * forward, loss, backward, slab reduction, gradient clip, Adam, post-step forward and KL of every epoch; row blocks of 16 run
 * forward -> loss -> input gradients without grid barriers, weight gradients are a second wave, an epoch costs 4 grid
 * barriers (5 in adapt mode).  It writes the same buffers and statistics as the launch chain it replaces
 * (sb200_mlp_forward_f32 + sb200_ppo_policy_loss_f32 / sb200_value_loss_f32 + sb200_linear_bwd_* +
 * sb200_grad_reduce_norm_f32 + sb200_clip_adam_f32 + sb200_ppo_kl_f32).
 *   sb200_epochs = the argument block of ONE optimiser: 3 layers ReLU-ReLU-any, no aux input, head <= 32 wide, widths <= 512.
 *   net->W / net->b must point INTO `params` (the flat buffer Adam updates); x_in/h1/h2/out/d1/d2/dpre are [M][ru4(width)]
 *   with zero padding columns (x_in receives the z-filtered input rows).
 *   mode 0 clip / 1 adapt (policy: out = tanh mean, log_var at params[extra_off..+A), early stop above stop_threshold),
 *   mode 2 value (MSE on `returns`).  grid: upper bound on the CTAs to launch (0: one per SM); cta_shift and workspace of the
 *   block are unused (the call takes the workspace).
 *   par != NULL with world > 1: data-parallel -- the KL scalar and the flat gradient are averaged over the ranks inside
 *   the kernel through the symmetric buffers of `par` (every rank must launch the same sequence). */
typedef struct {
    const sb200_mlp* net;
    float* params;
    int64_t n_params;
    int extra_off;
    const float* x;
    int64_t ldx;
    int M;
    const float* zf_stats;              /* NULL: no z-filter */
    double zf_eps;
    float *x_in, *h1, *h2, *out, *d1, *d2, *dpre;
    float* slabs;                       /* [splits][n_params] */
    int splits;
    float *grad, *exp_avg, *exp_avg_sq;
    const double* lr;
    double weight_decay;
    int clip_mode;
    double clip_value;
    void* opt_workspace;                /* sb200_optim_workspace_bytes(): holds the Adam step count */
    float* norm_out;                    /* optional: global gradient norm of the last step */
    int mode;
    const float* actions; int64_t lda;
    const float* adv;
    const float* behave_pd; int64_t ldb;
    const float* ref_pd; int64_t ldr;
    const float* returns;
    const double* hyper;                /* device: [clip_epsilon, beta] */
    double eta, kl_target, stop_threshold;
    float* stats;
    int* stop_flag;
    int epochs;
    void* workspace;                    /* unused (kept for layout) */
    int grid;
    int cta_shift;
    const sb200_par* par;
} sb200_epochs;
/* `policy` (mode 0 / 1) and `value` (mode 2, may be NULL) in one launch; `workspace` must hold
 * sb200_ppo_epochs2_workspace_bytes() bytes, 256-byte aligned, zero-initialised once.  Data-parallel: the two blocks must use
 * DIFFERENT sb200_par channels (both exchange in the same phase). */
int sb200_ppo_epochs2_supported(const sb200_epochs* policy, const sb200_epochs* value);
size_t sb200_ppo_epochs2_workspace_bytes(const sb200_epochs* policy, const sb200_epochs* value);
int sb200_ppo_epochs2_f32(const sb200_epochs* policy, const sb200_epochs* value, void* workspace, void* stream);
/* accumulated clock64 cycles per phase of the launches on `workspace` (2 x 16: CTA 0, last CTA; see epoch2.cu) */
int sb200_ppo_epochs2_profile(void* workspace, uint64_t* out32, int reset, void* stream);
int sb200_ppo_epochs2_cta_profile(void* workspace, uint64_t* out_192x8, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LSTM stem of RNN-mode PPO (csrc/lstm.cu; nn.LSTM(batch_first=True) of ppo_net.py:143-152,277-279,342-351; BPTT over
 * eff_len = n_step - horizon + 1 steps, ppo.py:389-406,507-525).  Gate order i, f, g, o; WhhT = [H][4H].
 *   rows_zfilter: out[b*L + t][0..D) = zfilter(x[b*batch_stride + t*row_stride + 0..D)) (plain gather if zf_stats NULL).
 *   lstm_forward: pre_x [B*L][4H] = x W_ih^T + b_ih (an MLP-kernel call); h0 / c0 row b at element b*ld_cells (NULL: zeros);
 *     h_out [B*L][ldh]; optional saves for the backward pass: h_prev (h_{t-1}, [B*L][ldh]), gates (post-activation), c_seq; optional
 *     final cells h_last / c_last [B][H].
 *   lstm_backward: dh_out [B*L][ldd] (gradient w.r.t. h_t) -> dpre [B*L][4H] (w.r.t. the gate pre-activations); the
 *     weight gradients are then sb200_linear_bwd_dw_f32(x, dpre) and sb200_linear_bwd_dw_f32(h_prev, dpre). */
int sb200_rows_zfilter_f32(const float* x, int64_t row_stride, int64_t batch_stride, int B, int L, int D,
                           const float* zf_stats, double eps, float* out, int64_t ldo, void* stream);
int sb200_lstm_forward_f32(const float* pre_x, const float* WhhT, const float* b_hh, const float* h0, const float* c0,
                           int64_t ld_cells, int B, int L, int H, int ldh, float* h_out, float* h_prev, float* gates,
                           float* c_seq, float* h_last, float* c_last, void* stream);
int sb200_lstm_backward_f32(const float* dh_out, int64_t ldd, const float* gates, const float* c_seq, const float* c0,
                            int64_t ld_cells, const float* WhhT, int B, int L, int H, float* dpre, void* stream);

/* Kernel family of the wide layers of sb200_mlp_forward_f32: 1 (default) = tensor-core mma.sync TF32 with the 3xTF32
 * error-compensated split (fp32-level accuracy, ~1e-6 relative) for batches above 2048 rows, fp32 FFMA below (where
 * the FFMA kernel is faster: 19 us vs 26 us at 1024 rows); 0 = fp32 FFMA kernels everywhere.  Env SB200_MMA overrides
 * the initial value. */
int sb200_set_forward_mode(int mode);

/* Backward of one Linear layer (kernel layout), replacing torch autograd in ppo.py:242,347 and
 * ddpg.py:306,330.
 *   dx: dX[M,K] = (dY[M,N] . W^T), multiplied by relu'(x_act) when x_act != NULL (x_act = the layer's
 *       saved post-ReLU input, so dX is directly the previous layer's pre-activation gradient).
 *   dw: `splits` partial slabs, slab z covering rows [z*rps, (z+1)*rps): dW_slabs + z*slab_stride is a
 *       [K][ldw] matrix, db_slabs + z*slab_stride a [ldw] vector (db_slabs may be NULL).  The slabs are
 *       summed in fixed order by sb200_grad_reduce_norm_f32 (deterministic, no atomics). */
int sb200_linear_bwd_dx_f32(const float* dY, int64_t ldy, const float* W, int ldw, const float* x_act,
                            int64_t ld_xact, float* dX, int64_t lddx, int M, int N, int K, void* stream);
int sb200_linear_bwd_dw_f32(const float* X, int64_t ldx, const float* dY, int64_t ldy, float* dW_slabs,
                            float* db_slabs, int64_t slab_stride, int splits, int ldw, int M, int K, int N,
                            void* stream);

/* ---------------------------------------------------------------------------------------------
 * Windowed GAE + n-step return (surreal/learner/ppo.py:372-374,387-418).
 *   rewards [B,n], values [B,n+1] (raw critic output; the (1-done) mask of ppo.py:387 is applied
 *   inside), dones [B,n].  horizon == n -> MLP branch (one output per window), horizon < n ->
 *   RNN branch (E = n-horizon+1 outputs per window).  adv/ret are [B,E].  norm_adv applies
 *   (adv-mean)/max(unbiased_std, 1e-4) over all B*E advantages.  rewards are multiplied by reward_scale
 *   (ppo.py:452) on load.
 *   workspace: sb200_gae_workspace_bytes() bytes, zero-initialised once by the caller. */
size_t sb200_gae_workspace_bytes(int B, int n, int horizon);
int sb200_gae_window_f32(const float* rewards, const float* values, const float* dones, int B, int n,
                         int horizon, double gamma, double lam, double reward_scale, int norm_adv, float* adv,
                         float* ret, void* workspace, void* stream);

/* pd[b] = [mean(A) | exp(log_var)(A) * exp(log_noise[b])]  (builders.py:127-129; per-actor noise of
 * ppo_agent.py:139 when log_noise != NULL). */
int sb200_make_pd_f32(const float* mean, int64_t ldm, const float* log_var, const float* log_noise, int B,
                      int A, float* pd, int64_t ldp, void* stream);
/* ZFilter.z_update (z_filter.py:44-57): stats = running_sum[D] | running_sumsq[D] | count[1], updated in place. */
int sb200_zfilter_update_f32(const float* x, int64_t ldx, int64_t rows, int D, float* stats, void* stream);

/* Global-batch statistics helpers for the data-parallel learner: moments3 = {sum, sum of squares, count} (fp64,
 * summed over ranks by the caller); normalize applies (x-mean)/max(unbiased std, floor) (ppo.py:413-416). */
int sb200_moments_f32(const float* x, int64_t n, double* moments3, void* stream);
int sb200_normalize_f32(float* x, int64_t n, const double* moments3, double floor_value, void* stream);
int sb200_add_f32(float* dst, const float* src, int64_t n, void* stream);
/* RewardFilter as called from ppo.py:452-456: out = forward(rewards*reward_scale) with the current statistics,
 * then update (running_sumsq is OVERWRITTEN, reward_filter.py:42).  stats = count | running_sum | running_sumsq. */
int sb200_reward_filter_f32(const float* rewards, int64_t n, double reward_scale, double eps, float* stats,
                            float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * PPO losses: forward + gradient in one pass (replaces surreal/learner/ppo.py:194-225, 250-285,
 * 311-332, 553-557, 568-575 and DiagGauss of surreal/model/ppo_net.py:29-72 with torch autograd).
 * stats[] is a device float array of SB200_STAT_COUNT slots. */
#define SB200_STAT_SURR 0            /* _surr_loss */
#define SB200_STAT_LOSS 1            /* _clip_surr_loss (clip) / _kl_loss_adapt (adapt) */
#define SB200_STAT_ENTROPY 2         /* _entropy */
#define SB200_STAT_KL_PRE 3          /* adapt: _pol_kl inside the loss (before the step) */
#define SB200_STAT_KL_POST 4         /* _pol_kl after the step (early-stop test, ppo.py:553-556) */
#define SB200_STAT_GRAD_NORM_ACTOR 5
#define SB200_STAT_VAL_LOSS 6
#define SB200_STAT_EXPLAINED_VAR 7
#define SB200_STAT_GRAD_NORM_CRITIC 8
#define SB200_STAT_RETURN_MEAN 9     /* _avg_return_targ */
#define SB200_STAT_LOG_SIG 10        /* _avg_log_sig */
#define SB200_STAT_BEHAVE_LIK 11     /* _avg_behave_likelihood */
#define SB200_STAT_IS_WEIGHT 12      /* _avg_is_weight */
#define SB200_STAT_REF_BEHAVE_KL 13  /* _ref_behave_diff */
#define SB200_STAT_EPOCHS 14         /* number of policy epochs executed this learn() */
#define SB200_STAT_VAL_MOMENTS 16    /* 8 slots: mean(ret-v), mean((ret-v)^2), mean(ret), mean(ret^2) as (hi, lo) float pairs */
#define SB200_STAT_COUNT 32

size_t sb200_ppo_loss_workspace_bytes(int B, int A);   /* zero-initialise once */
/* mode 0 = clip (hyper[0] = clip_epsilon), mode 1 = adapt (hyper[1] = beta; needs sb200_ppo_kl_f32(ref, learn)
 * to have run on the same workspace first).  mean: actor output after tanh [B,ldm]; dpre: gradient w.r.t.
 * the pre-tanh output [B,ldd] (padding columns zeroed); dlog_var [A].  hyper is a DEVICE array of doubles so
 * that publish-time adaptation (ppo.py:648-661) does not invalidate captured graphs.
 * stop_flag (may be NULL): when *stop_flag != 0 the kernel is a no-op (device-side KL early stop). */
int sb200_ppo_policy_loss_f32(int mode, const float* mean, int64_t ldm, const float* log_var,
                              const float* actions, int64_t lda, const float* adv, const float* behave_pd,
                              int64_t ldb, const float* ref_pd, int64_t ldr, int B, int A,
                              const double* hyper, double eta, double kl_target, float* dpre, int64_t ldd,
                              float* dlog_var, float* stats, void* workspace, const int* stop_flag, void* stream);
/* mean KL(p0 || (mean, exp(log_var))) -> stats[stat_slot] (slot < 0: none) and the workspace; raises *stop_flag
 * when the mean exceeds stop_threshold (> 0). */
int sb200_ppo_kl_f32(const float* p0, int64_t ld0, const float* mean, int64_t ldm, const float* log_var,
                     int B, int A, float* stats, int stat_slot, double stop_threshold, int* stop_flag,
                     int defer, void* workspace, void* stream);
/* Data-parallel split of the above: with defer != 0 sb200_ppo_kl_f32 only leaves the LOCAL mean KL as a double at
 * byte offset sb200_ppo_loss_kl_offset() of the workspace; the caller averages it over ranks (NCCL) and then
 * sb200_ppo_kl_apply publishes it to stats / raises the stop flag identically on every rank. */
int sb200_ppo_kl_apply(void* workspace, float* stats, int stat_slot, double stop_threshold, int* stop_flag,
                       void* stream);
size_t sb200_ppo_loss_kl_offset(void);
int sb200_value_loss_f32(const float* values, int64_t ldv, const float* returns, int B, float* dpre,
                         int64_t ldd, float* stats, void* workspace, void* stream);
int sb200_ppo_final_stats_f32(const float* mean, int64_t ldm, const float* log_var, const float* actions,
                              int64_t lda, const float* behave_pd, int64_t ldb, const float* ref_pd,
                              int64_t ldr, int B, int A, float* stats, void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimiser over one flat parameter buffer (replaces clip_grad_norm_/clip_grad_value_ + torch.optim.Adam:
 * ppo.py:159-168,244-247,349-352; ddpg.py:145-165,309-310,332-333).
 *   grad_reduce_norm: grad[i] = scale * sum_z slabs[z*slab_stride + i] (fixed order); global L2 norm (and
 *                     step += 1 when bump_step) into the workspace.  Data-parallel learners call it twice around
 *                     the NCCL all-reduce: (slabs -> grad, scale 1, no bump), (grad -> grad, 1/world, bump).
 *   clip_adam: clip_mode 0 none / 1 global norm (clip_value = max_norm) / 2 by value; lr is a DEVICE double.
 *   workspace: sb200_optim_workspace_bytes(), zero-initialised once (it holds the Adam step count). */
size_t sb200_optim_workspace_bytes(void);
int sb200_grad_reduce_norm_f32(const float* slabs, int64_t slab_stride, int splits, float* grad, int64_t n,
                               double scale, int bump_step, void* workspace, const int* stop_flag, void* stream);
int sb200_clip_adam_f32(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                        const double* lr, double beta1, double beta2, double eps, double weight_decay,
                        int clip_mode, double clip_value, void* workspace, float* norm_out,
                        const int* stop_flag, void* stream);
/* target = target*(1-tau) + tau*src (soft target update, ddpg.py:410-418); a no-op when *stop_flag != 0. */
int sb200_soft_update_f32(float* target, const float* src, int64_t n, double tau, const int* stop_flag, void* stream);

/* ---------------------------------------------------------------------------------------------
 * DDPG element-wise pieces (surreal/learner/ddpg.py:261-262,279,305,324-331,335-341); the networks run through
 * sb200_mlp_forward_f32 (critic: aux_layer = 1 for cat(h, action)) and the backward / optimiser entries above. */
#define SB200_DSTAT_ACTOR_LOSS 0
#define SB200_DSTAT_CRITIC_LOSS 1
#define SB200_DSTAT_ACTION_NORM 2
#define SB200_DSTAT_REWARDS 3
#define SB200_DSTAT_Q_TARGET 4
#define SB200_DSTAT_Q_POLICY 5
#define SB200_DSTAT_ACTION_ABSMAX 6   /* for the deferred `assert |a| <= 1` of ddpg.py:261-262 */
/* byte offset inside the DDPG workspace of the int32 "bad action" flag: sb200_ddpg_target*_f32 set it to 1 when
 * max|a| > 1 (the reference asserts this BEFORE any update, ddpg.py:261-262); pass its address as stop_flag to the
 * optimiser / soft-update calls of the same learn() so an out-of-range batch leaves every parameter untouched. */
size_t sb200_ddpg_bad_action_offset(void);
size_t sb200_ddpg_workspace_bytes(int B);
/* y = rewards + discount * q_next * (1 - dones), discount = gamma ** n_step. */
int sb200_ddpg_target_f32(const float* rewards, const float* q_next, int64_t ldq, const float* dones,
                          const float* actions, int64_t lda, int B, int A, double discount, float* y,
                          float* stats, void* workspace, void* stream);
/* MSE(q, y): dq = 2 (q - y) / B. */
int sb200_ddpg_critic_loss_f32(const float* q, int64_t ldq, const float* y, int B, float* dq, int64_t ldd,
                               float* stats, void* workspace, void* stream);
/* TD3 options (ddpg.py:267-283): target2 = ddpg_target with y = min(y, y2) over two target critics; smooth_action =
 * clamp(pi + clip(policy_noise * N(0,1), -noise_clip, noise_clip), -1, 1) (unit_noise [B][A] injected draws, or NULL
 * for Philox keyed by (seed, *step_counter, row)). */
int sb200_ddpg_target2_f32(const float* rewards, const float* q_next, int64_t ldq, const float* q_next2, int64_t ldq2,
                           const float* dones, const float* actions, int64_t lda, int B, int A, double discount,
                           float* y, float* stats, void* workspace, void* stream);
int sb200_ddpg_smooth_action_f32(const float* pi, int64_t ldp, const float* unit_noise, int B, int A,
                                 double policy_noise, double noise_clip, uint64_t seed, const uint64_t* step_counter,
                                 float* out, int64_t ldo, void* stream);
/* actor loss -mean(q_pi): seeds dq = -1/B for the backward pass through the critic. */
int sb200_ddpg_actor_seed_f32(const float* q_pi, int64_t ldq, int B, float* dq, int64_t ldd, float* stats,
                              void* workspace, void* stream);
/* dpre = dout * (1 - out^2). */
int sb200_tanh_bwd_f32(const float* dout, int64_t ldo, const float* out, int64_t ldy, int B, int A,
                       float* dpre, int64_t ldd, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched actors (one call serves all N co-located actors of a step).
 *   ppo_sample: PPOAgent.act after the network (surreal/agent/ppo_agent.py:138-149): pd = [mean | exp(log_var)*
 *     exp(log_noise_i)], action = clip(eps*std+mean, -1, 1).  eps [N,A] injected N(0,1) draws or NULL for
 *     Philox4x32-10 keyed by (seed, *step_counter, actor).  When stage_act != NULL the step's action / pd rows
 *     are also written to the window staging area at stage_pos[i] (see ppo_window_step).
 *   ddpg_noise: DDPGAgent.act after the network (ddpg_agent.py:176-183): clip -> + sigma_i*N(0,1) -> clip. */
int sb200_ppo_sample_f32(const float* mean, int64_t ldm, const float* log_var, const float* log_noise,
                         const float* eps, int N, int A, int deterministic, uint64_t seed,
                         const uint64_t* step_counter, float* action, float* pd, const int* stage_pos,
                         float* stage_act, float* stage_pd, int n_step, void* stream);
/*   ppo_sample_assign: ppo_sample fused with the slot assignment of ppo_window_step for the windows this step
 *     completes (it depends only on the deque lengths, so it can precede the env step): writes dest[N]
 *     (slot | -1 not complete | -2 complete but dropped), advances fifo_state and *step_counter (+1, after every
 *     block has drawn with the old value).  Follow with ppo_window_step(slots_assigned=1) or
 *     synth_env_window_step. */
int sb200_ppo_sample_assign_f32(const float* mean, int64_t ldm, const float* log_var, const float* log_noise,
                                const float* eps, int N, int A, int deterministic, uint64_t seed,
                                uint64_t* step_counter, float* action, float* pd, const int* stage_pos,
                                float* stage_act, float* stage_pd, int n_step, void* fifo_state, int* dest,
                                void* stream);
int sb200_ddpg_noise_f32(const float* mean, int64_t ldm, const float* sigma, const float* unit_noise, int N,
                         int A, int deterministic, uint64_t seed, const uint64_t* step_counter,
                         float* action, void* stream);
/*   ddpg_ou_noise: the same with Ornstein-Uhlenbeck exploration (surreal/agent/action_noise.py:22-39): ou_state [N][A]
 *     float64 is advanced in place, x <- x + theta*(0 - x)*dt + sigma_i*sqrt(dt)*N(0,1); sigma [N] float64.  The caller
 *     zeroes ou_state at episode start (DDPGAgent.pre_episode, ddpg_agent.py:205-208). */
int sb200_ddpg_ou_noise_f32(const float* mean, int64_t ldm, const double* sigma, const float* unit_noise, int N, int A,
                            int deterministic, uint64_t seed, const uint64_t* step_counter, double theta, double dt,
                            double* ou_state, float* action, void* stream);
/* Synthetic device-resident environment of the benchmark configs (SURVEY §8d): s' = tanh(Ws s + Wa a) + 0.01 xi,
 * r = -|s|^2/D + 0.1 xi', done at max_steps (MaxStepWrapper, env/wrapper.py:142-163) with auto-reset.
 * state [N,D] is updated in place to what the agent observes next; obs_next is the true successor.
 * Ws / Wa are passed transposed (k-major): WsT [D][D] with WsT[k][d] = Ws[d][k], WaT [A][D]. */
int sb200_synth_env_step_f32(float* state, const float* action, const float* Ws, const float* Wa, int N,
                             int D, int A, int max_steps, int* ep_step, uint64_t seed,
                             const uint64_t* step_counter, float* obs_next, float* reward, float* done,
                             void* stream);
/* synth_env_step fused with the commit half of ppo_window_step (dest from ppo_sample_assign): the successor
 * state is staged straight from shared memory.  One launch per rollout step instead of three. */
int sb200_synth_env_window_step_f32(float* state, const float* action, const float* Ws, const float* Wa, int N,
                                    int D, int A, int max_steps, int* ep_step, uint64_t seed,
                                    const uint64_t* step_counter, float* obs_next, float* reward, float* done,
                                    int n_step, int stride, int* stage_pos, float* stage_obs, float* stage_act,
                                    float* stage_pd, float* stage_rew, float* stage_done, const int* dest,
                                    float* r_obs, float* r_act, float* r_pd, float* r_rew, float* r_done,
                                    void* stream);

/* Host-env fast path (one C call per agent.act() / ExpSender-wrapper step when the environment lives on the host):
 *   ppo_act_host: [H2D obs_host -> obs_dev unless obs_host is NULL] -> policy forward -> ppo_sample (ppo_sample_assign
 *     when fifo_state != NULL) -> D2H action / pd -> ONE stream synchronisation.  Host pointers must be pinned.
 *   ppo_window_step_host: H2D of the step's successor / next observation, reward and done, then ppo_window_step. */
int sb200_ppo_act_host_f32(const sb200_mlp* net, const sb200_zfilter* zf, const float* obs_host, float* obs_dev, int N,
                           float* mean_dev, const float* log_var, const float* log_noise, int deterministic,
                           uint64_t seed, uint64_t* step_counter, float* action_dev, float* pd_dev,
                           const int* stage_pos, float* stage_act, float* stage_pd, int n_step, void* fifo_state,
                           int* dest, float* action_host, float* pd_host, void* stream);
int sb200_ppo_window_step_host_f32(const float* obs_next_host, const float* obs_reset_host, const float* reward_host,
                                   const float* done_host, float* obs_next_dev, float* obs_reset_dev,
                                   float* reward_dev, float* done_dev, int N, int n_step, int stride, int D, int A,
                                   int* stage_pos, float* stage_obs, float* stage_act, float* stage_pd,
                                   float* stage_rew, float* stage_done, int* dest_scratch, void* fifo_state,
                                   float* r_obs, float* r_act, float* r_pd, float* r_rew, float* r_done,
                                   uint64_t* step_counter, int slots_assigned, void* stream);

/* Persistent rollout: T steps of policy forward -> sample -> synthetic env step -> window staging for ALL N
 * actors in ONE launch (a 4-CTA cluster owns 32 actors for the whole chunk; the policy weights stay resident in
 * shared memory, layer outputs cross CTAs through distributed shared memory).  Replaces T x (ppo_sample_assign +
 * synth_env_window_step + the policy forward), i.e. the actor main loop of surreal/agent/base.py:224-271 for a
 * device-resident env.  Same sampling / env arithmetic and Philox keys as the per-step entries.
 *   Completed windows are written to a per-actor OUTBOX (o_*: [N*W] records in the replay's record layout,
 *   ev_step [N*W] = chunk-relative completion step, ev_count [N]); W >= T / stride + 2.
 *   rollout_commit then assigns FIFO slots in the reference's (step, actor) arrival order, copies the windows into
 *   the replay ring, advances fifo_state and *step_counter (+T).  scratch: sb200_ppo_rollout_scratch_ints() ints.
 *   rollout_supported: 1 when `net` (2 hidden layers whose widths are multiples of 16, head <= 32, D % 4 == 0,
 *   D <= 128) fits the shared-memory plan; otherwise use the per-step entries. */
typedef struct {
    const sb200_mlp* net;               /* policy: D -> H1 -> H2 -> A */
    const float* zf_stats;              /* NULL: no z-filter */
    float zf_eps;
    const float* log_var;               /* [A] */
    const float* log_noise;             /* [N] or NULL */
    uint64_t agent_seed;
    int deterministic;
    float* state;                       /* [N][D] env state = next observation, updated in place */
    const float* WsT;                   /* [D][D] k-major */
    const float* WaT;                   /* [A][D] k-major */
    int* ep_step;                       /* [N] */
    int max_steps;
    uint64_t env_seed;
    float* action;                      /* outputs of the LAST step, like the per-step entries leave them */
    float* pd;
    float* obs_next;
    float* reward;
    float* done;
    int* stage_pos;                     /* window staging, see ppo_window_step */
    float* stage_obs;
    float* stage_act;
    float* stage_pd;
    float* stage_rew;
    float* stage_done;
    float* o_obs;                       /* outbox */
    float* o_act;
    float* o_pd;
    float* o_rew;
    float* o_done;
    int* ev_step;
    int* ev_count;
    int W;
    int N, D, A, n_step, stride, T;
    const uint64_t* step_counter;       /* read only; rollout_commit advances it */
} sb200_ppo_rollout;
int sb200_ppo_rollout_supported(const sb200_mlp* net, int D, int A);
size_t sb200_ppo_rollout_scratch_ints(int N, int W, int T);
int sb200_ppo_rollout_f32(const sb200_ppo_rollout* args, void* stream);
int sb200_ppo_rollout_commit_f32(const sb200_ppo_rollout* args, int* scratch, void* fifo_state, float* r_obs,
                                 float* r_act, float* r_pd, float* r_rew, float* r_done, uint64_t* step_counter,
                                 void* stream);

/* ---------------------------------------------------------------------------------------------
 * Experience staging + HBM replay.
 *   ppo_window_step: ExpSenderWrapperMultiStepMovingWindowWithInfo._step (exp_sender_wrapper.py:209-228) for N
 *     actors + FIFOReplay.insert (fifo_replay.py:27,34-35): per-actor deque in HBM (stage_*: obs [N][n+1][D],
 *     act [N][n][A], pd [N][n][2A], rew/done [N][n], pos [N]); completed windows are copied into FIFO slots in
 *     (step, actor) order, drop-oldest at capacity; `stride` items are popped; done clears the deque.
 *     Replay storage r_*: obs [C][n+1][D] (row n = obs_next), act [C][n][A], pd [C][n][2A], rew/done [C][n].
 *   fifo_state: sb200_fifo_state_bytes() bytes {int head,count,capacity,dropped; int64 total_in,total_out}.
 *   fifo_pop: FIFOReplay.sample (fifo_replay.py:37-39): slot ids of the `batch` oldest windows; *status = 1
 *     if fewer are queued.   fifo_push: host-side Replay.insert() of k windows -> their slot ids.
 *   replay_gather: out[b] = src[idx[b]] for records of record_floats floats (idx32 or idx64 non-NULL). */
size_t sb200_fifo_state_bytes(void);
int sb200_ppo_window_step_f32(const float* obs_next, const float* obs_reset, const float* reward,
                              const float* done, int N, int n_step, int stride, int D, int A,
                              int* stage_pos, float* stage_obs, float* stage_act, float* stage_pd,
                              float* stage_rew, float* stage_done, int* dest_scratch, void* fifo_state,
                              float* r_obs, float* r_act, float* r_pd, float* r_rew, float* r_done,
                              uint64_t* step_counter, int slots_assigned, void* stream);
int sb200_fifo_pop(void* fifo_state, int batch, int* idx, int* status, void* stream);
int sb200_fifo_push(void* fifo_state, int k, int* slots, void* stream);
int sb200_replay_gather_f32(const float* src, int64_t record_floats, const int* idx32, const int64_t* idx64,
                            int batch, float* out, void* stream);
/* Every field of the sampled records in ONE launch (srcs / outs / record_floats are HOST arrays of nfields <= 8 entries):
 * outs[f][b] = srcs[f][idx[b]].  Replaces the per-key np.stack loops of aggregator.py:52-103,151-205. */
int sb200_replay_gather_multi_f32(const float* const* srcs, float* const* outs, const int64_t* record_floats,
                                  int nfields, const int* idx32, const int64_t* idx64, int batch, void* stream);
/*   ssar_step: ExpSenderWrapperSSARNStepBootstrap._step (exp_sender_wrapper.py:96-112) for N actors +
 *     UniformReplay.insert (uniform_replay.py:36-41): k-th insert -> slot k % capacity, actor order.
 *     uniform_state: sb200_uniform_state_bytes() bytes {int64 next_idx,size,capacity,total_in}. */
size_t sb200_uniform_state_bytes(void);
int sb200_ssar_step_f32(const float* obs, const float* action, const float* obs_next, const float* reward,
                        const float* done, int N, int n_step, double gamma, int D, int A, int* dq_len,
                        float* dq_obs, float* dq_act, double* dq_rew, int* dest_scratch, float* emit_scratch,
                        void* uniform_state, float* r_obs, float* r_obs_next, float* r_act, float* r_rew,
                        float* r_done, uint64_t* step_counter, void* stream);
/* CPython random.Random-compatible MT19937 on the HOST (uniform_replay.py:43-45 draws
 * random.randint(0, len-1) per sample; SURVEY Appendix A.6).  state_h: sb200_mt19937_state_bytes() bytes. */
size_t sb200_mt19937_state_bytes(void);
int sb200_mt19937_seed_h(void* state_h, const uint32_t* key_h, int key_len);     /* random.seed(int): 32-bit limbs */
int sb200_mt19937_set_state_h(void* state_h, const uint32_t* words624_h, int index);   /* random.getstate()[1] */
int sb200_mt19937_get_state_h(const void* state_h, uint32_t* words624_h, int* index);
int sb200_mt19937_randint_fill_h(void* state_h, int64_t population, int64_t count, int64_t* out_h);

#ifdef __cplusplus
}
#endif
#endif /* SURREAL_B200_H */
