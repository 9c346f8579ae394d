/*
 * hpc_rll_b200.h -- C ABI of the B200-native trajectory-return library (libhpc_rll_b200.so).
 *
 * Drop-in boundary for DI-hpc's `hpc_rl_utils` native extension
 * (/root/reference/src/rl_utils/entry.cpp:8-39, declarations in
 * /root/reference/include/hpc/rll/cuda/rl_utils/entry.h:62-165).  The reference boundary is C++
 * (`std::vector<torch::Tensor>` in/out); here every entry point is plain C: device pointers, sizes,
 * scalars and a CUDA stream handle -- no torch types -- so it can be bound from ctypes / pybind /
 * cgo alike.  INTEGRATION.md shows the binding used by `hpc_rll.rl_utils`.
 *
 * Conventions
 *   - all tensors are fp32, row-major, resident on the CURRENT CUDA device; `action` tensors int64
 *   - (T,B) means T rows of B contiguous columns (time-major, as in the reference)
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream)
 *   - every function returns HPC_RLL_OK (0) or an error code; hpc_rll_last_error() gives the text
 *   - `global_B`: the batch may be one shard of a data-parallel global batch; mean-type losses and
 *     their gradients are normalised by the GLOBAL element count (0 means "B is the whole batch").
 *     Per-rank losses then add up (one all-reduce(SUM)) to the global loss.
 *   - gamma/lambda/... are doubles: the reference's Python layer computes e.g. gamma*lambda and
 *     gamma**nstep in double before the value meets an fp32 tensor (hpc_rll/origin/gae.py:30)
 *   - `workspace`: caller-provided device scratch of at least hpc_rll_workspace_bytes(op, ...) bytes
 *   - nothing here synchronises the device or the stream; no CPU fallback exists.
 */
#ifndef HPC_RLL_B200_H_
#define HPC_RLL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HPC_RLL_OK 0
#define HPC_RLL_EINVAL 1 /* bad argument (null pointer, negative size, misaligned ...) */
#define HPC_RLL_ECUDA 2  /* a CUDA runtime/driver call failed */
#define HPC_RLL_ENOSUP 3 /* unsupported configuration */

/* op ids for hpc_rll_workspace_bytes / hpc_rll_debug_set_config */
#define HPC_RLL_OP_GAE 0
#define HPC_RLL_OP_TD_LAMBDA 1
#define HPC_RLL_OP_VTRACE 2
#define HPC_RLL_OP_UPGO 3
#define HPC_RLL_OP_PPO 4
#define HPC_RLL_OP_Q_NSTEP_TD 5
#define HPC_RLL_OP_DIST_NSTEP_TD 6
#define HPC_RLL_OP_QRDQN_NSTEP_TD 7
#define HPC_RLL_OP_IQN_NSTEP_TD 8
#define HPC_RLL_OP_GAE_MOMENTS 9 /* workspace sizing only; tuning follows HPC_RLL_OP_GAE */
#define HPC_RLL_OP_SCATTER_CONNECTION 10 /* no workspace; tuning: bit 0 forward thread stores, bit 1 backward gather */
#define HPC_RLL_OP_COUNT 11

/* ---- library ------------------------------------------------------------------------------ */
const char* hpc_rll_version(void);
const char* hpc_rll_last_error(void); /* thread-local, valid until the next failing call */
/* number of CUDA kernels this library has launched in this process (bench.py: "gpu_launches") */
uint64_t hpc_rll_launch_count(void);
/* scratch bytes an op needs for sizes (T,B,N); N = action dim / n_atom / tau as relevant */
size_t hpc_rll_workspace_bytes(int op, int64_t T, int64_t B, int64_t N);
/* tuning/debug: force kernel configuration `cfg` for `op` (-1 = automatic) */
int hpc_rll_debug_set_config(int op, int cfg);

/* out[i] = a[0]*x[i] + b[0]*y[i]  (a, b DEVICE scalars; b and y may be NULL together: out = a[0]*x).  Glue for
 * the legacy `hpc_rl_utils` tensor-list shim (di_hpc_b200/csrc_torch/legacy.cpp), whose backward entry points
 * (/root/reference/src/rl_utils/entry.cpp:24-38) receive only buffers that are linear in the upstream gradients. */
int hpc_rll_axpby(const float* a, const float* x, const float* b, const float* y, float* out, int64_t n,
                  void* stream);

/* ---- GAE ------------------------------------------------------------------------------------
 * replaces GaeForward (/root/reference/src/rl_utils/gae.cu:8-28, kernel
 * include/hpc/rll/cuda/rl_utils/gae_kernel.h:10-29); semantics of hpc_rll/origin/gae.py:28-37.
 *   value (T+1,B), reward (T,B) -> adv (T,B).
 * hpc_rll_gae_backward is the adjoint the reference lacks (GAEFunction.backward returns None,
 * hpc_rll/rl_utils/gae.py:16-18):  grad_adv (T,B) -> grad_value (T+1,B), grad_reward (T,B).
 * The *_ld variants take row pitches in elements (>= B) for strided views. */
int hpc_rll_gae_forward(const float* value, const float* reward, float* adv, int64_t T, int64_t B, double gamma,
                        double lambda, void* stream);
int hpc_rll_gae_backward(const float* grad_adv, float* grad_value, float* grad_reward, int64_t T, int64_t B,
                         double gamma, double lambda, void* stream);
int hpc_rll_gae_forward_ld(const float* value, int64_t ld_value, const float* reward, int64_t ld_reward,
                           float* adv, int64_t ld_adv, int64_t T, int64_t B, double gamma, double lambda,
                           void* stream);
int hpc_rll_gae_backward_ld(const float* grad_adv, int64_t ld_grad_adv, float* grad_value, int64_t ld_grad_value,
                            float* grad_reward, int64_t ld_grad_reward, int64_t T, int64_t B, double gamma,
                            double lambda, void* stream);
/* GAE forward that also returns the raw moments of the advantages it writes:
 *   moments[0] = sum(adv), moments[1] = sum(adv^2)   (fp64, device memory, fixed summation order; each
 *   column folds fp32 runs of 16 rows into fp64 accumulators)
 * for the normalisation (adv - adv.mean()) / (adv.std() + 1e-8) that precedes ppo_error
 * (/root/reference/hpc_rll/origin/ppo.py:43-47) -- fused here so that `adv` is not re-read twice for
 * mean and std.  Data-parallel callers all-reduce(SUM) `moments` before hpc_rll_adv_stats.
 * value/reward/adv contiguous.  Workspace: hpc_rll_workspace_bytes(HPC_RLL_OP_GAE_MOMENTS, T, B, 0). */
int hpc_rll_gae_forward_moments(const float* value, const float* reward, float* adv, double* moments, int64_t T,
                                int64_t B, double gamma, double lambda, void* workspace, size_t workspace_bytes,
                                void* stream);
/* moments (device, fp64) over `count` elements -> stats[0] = mean, stats[1] = unbiased std + 1e-8
 * (device, fp32; exactly the two scalars of the normalisation above).  count == 1 gives NaN like torch.std.
 * count <= 0: the element count is read from moments[2] (a caller-filled third double, so that sums and
 * count travel through one all-reduce and no host round trip is needed). */
int hpc_rll_adv_stats(const double* moments, int64_t count, float* stats, void* stream);
/* T-CHUNKED scan (round 2): rows [t0, t0+rows) of a T_total-row problem, the scan state carried in `carry`
 * (2,B) fp32 on the device.  Bit-identical to the monolithic call (the per-column recurrence is sequential; chunking
 * does not re-associate it).  This is what lets a (T,B) problem be streamed through the device as contiguous row
 * ranges (hpc_rll_gae_fwd_bwd_host) or produced/consumed chunk by chunk by a rollout collector.
 *   forward : chunks are processed from the LAST one to the first.  carry[0:B] = g (0 before the first call),
 *             carry[B:2B] = the value row that follows the chunk (value[T_total] before the first call); on return
 *             g at row t0 and value row t0.  value/reward/adv are (rows,B) (no extra value row).
 *   backward: chunks are processed from the FIRST one to the last.  carry = (ghat, dd of the previous row), zeros
 *             before the first call.  grad_value is (rows,B), plus row `rows` (= global row T_total) in the call
 *             with t0 + rows == T_total.
 * t0 must be even for the TMA path (else a generic CUDA kernel runs). */
int hpc_rll_gae_forward_chunk(const float* value, const float* reward, float* adv, float* carry, int64_t T_total,
                              int64_t t0, int64_t rows, int64_t B, double gamma, double lambda, void* stream);
int hpc_rll_gae_backward_chunk(const float* grad_adv, float* grad_value, float* grad_reward, float* carry,
                               int64_t T_total, int64_t t0, int64_t rows, int64_t B, double gamma, double lambda,
                               void* stream);
/* HOST-buffer entry (end-to-end path): pinned (or pageable) host arrays in, host arrays out.  Runs forward and
 * backward on the current device as a T-chunked carry pipeline: contiguous row ranges stream over the H2D engine,
 * full-width kernels, the D2H engine drains results, all overlapped on internal streams (a pool of pipes: concurrent
 * callers do not serialise); returns after all results have landed in the host buffers (sleeping, not spinning).
 * Any of h_grad_adv/h_grad_value/h_grad_reward may be NULL together (forward only).
 * Tuning: HPC_RLL_HOST_CHUNK_ROWS (rows per stage, multiple of 4; default ~4 MB per tensor per stage). */
int hpc_rll_gae_fwd_bwd_host(const float* h_value, const float* h_reward, const float* h_grad_adv, float* h_adv,
                             float* h_grad_value, float* h_grad_reward, int64_t T, int64_t B, double gamma,
                             double lambda);

/* test hook: the stage heights hpc_rll_gae_fwd_bwd_host would use for a (T,B) problem (host-only, no CUDA call);
 * writes up to `cap` entries, returns the number of stages */
int64_t hpc_rll_debug_host_schedule(int64_t T, int64_t B, int64_t* rows, int64_t cap);

/* ---- host placement (NUMA) --------------------------------------------------------------------
 * A B200 box has its GPUs split over two CPU sockets; host buffers that feed a GPU over PCIe should live on that
 * GPU's socket, or eight ranks push all their DMA traffic through one socket's DRAM and the inter-socket link.
 *   hpc_rll_device_numa_node     NUMA node of CUDA device `device` (sysfs numa_node of its PCI function), -1 unknown
 *   hpc_rll_bind_thread_to_device  restrict the CALLING thread to that node's CPUs (threads it spawns inherit it)
 *                                and prefer that node for its page allocations; returns the node or -1 (left as is).
 *                                device < 0 undoes it (affinity from before the first bind, default memory policy)
 *   hpc_rll_host_alloc / _free   page-locked host memory (cudaHostAlloc) allocated and first touched while the calling
 *                                thread is confined to that node (its affinity / policy are restored afterwards) */
int hpc_rll_device_numa_node(int device);
int hpc_rll_bind_thread_to_device(int device);
void* hpc_rll_host_alloc(size_t bytes, int device);
int hpc_rll_host_free(void* ptr);

/* ---- TD(lambda) ----------------------------------------------------------------------------
 * replaces TdLambdaForward / TdLambdaBackward (/root/reference/src/rl_utils/td_lambda.cu:8-52, kernels
 * include/hpc/rll/cuda/rl_utils/td_lambda_kernel.h:11-51); semantics of hpc_rll/origin/td.py:148-176.
 *   forward : value (T+1,B), reward (T,B), weight (T,B) or NULL (= ones)
 *             -> loss[1] = 0.5*mean(w*(ret-v)^2),  grad_buf (T,B) = dloss/dvalue[:T] (no upstream grad)
 *   backward: grad_loss[1] (device), grad_buf -> grad_value (T+1,B) (row T is zero) */
int hpc_rll_td_lambda_forward(const float* value, const float* reward, const float* weight, float* loss,
                              float* grad_buf, int64_t T, int64_t B, double gamma, double lambda,
                              int64_t global_B, void* workspace, size_t workspace_bytes, void* stream);
int hpc_rll_td_lambda_backward(const float* grad_loss, const float* grad_buf, float* grad_value, int64_t T,
                               int64_t B, void* stream);

/* ---- V-trace --------------------------------------------------------------------------------
 * replaces VTraceForward / VTraceBackward (/root/reference/src/rl_utils/vtrace.cu:8-130, kernels
 * include/hpc/rll/cuda/rl_utils/vtrace_kernel.h:11-273); semantics of hpc_rll/origin/vtrace.py:63-79.
 *   forward : target_output, behaviour_output (T,B,N); action (T,B) int64; value (T+1,B); reward (T,B);
 *             weight (T,B) or NULL -> losses[3] = {policy, value, entropy};
 *             saved for backward: pg_coef (T,B) = -adv*w/n, gv_buf (T,B) = 2(v-ret)w/n   (n = T*global_B)
 *   backward: three upstream gradients (device scalars) -> grad_target_output (T,B,N), grad_value (T+1,B) */
int hpc_rll_vtrace_forward(const float* target_output, const float* behaviour_output, const int64_t* action,
                           const float* value, const float* reward, const float* weight, float* losses,
                           float* pg_coef, float* gv_buf, int64_t T, int64_t B, int64_t N, double gamma,
                           double lambda, double rho_clip_ratio, double c_clip_ratio, double rho_pg_clip_ratio,
                           int64_t global_B, void* workspace, size_t workspace_bytes, void* stream);
int hpc_rll_vtrace_backward(const float* grad_policy_loss, const float* grad_value_loss,
                            const float* grad_entropy_loss, const float* target_output, const int64_t* action,
                            const float* weight, const float* pg_coef, const float* gv_buf, float* grad_target_output,
                            float* grad_value, int64_t T, int64_t B, int64_t N, int64_t global_B, void* stream);

/* ---- UPGO -----------------------------------------------------------------------------------
 * replaces UpgoForward / UpgoBackward (/root/reference/src/rl_utils/upgo.cu:8-69, kernels
 * include/hpc/rll/cuda/rl_utils/upgo_kernel.h:11-108); semantics of hpc_rll/origin/upgo.py:40-70.
 *   forward : target_output (T,B,N); rhos (T,B); action (T,B) int64; rewards (T,B); bootstrap_values (T+1,B)
 *             -> loss[1]; saved for backward: coef (T,B) = -adv/n
 *   backward: grad_loss (device scalar) -> grad_target_output (T,B,N) */
int hpc_rll_upgo_forward(const float* target_output, const float* rhos, const int64_t* action,
                         const float* rewards, const float* bootstrap_values, float* loss, float* coef, int64_t T,
                         int64_t B, int64_t N, int64_t global_B, void* workspace, size_t workspace_bytes,
                         void* stream);
int hpc_rll_upgo_backward(const float* grad_loss, const float* target_output, const int64_t* action,
                          const float* coef, float* grad_target_output, int64_t T, int64_t B, int64_t N,
                          void* stream);

/* ---- PPO ------------------------------------------------------------------------------------
 * replaces PPOForward / PPOBackward (/root/reference/src/rl_utils/ppo.cu:8-111, kernels
 * include/hpc/rll/cuda/rl_utils/ppo_kernel.h:12-283); semantics of hpc_rll/origin/ppo.py:51-80.
 *   forward : logits_new, logits_old (B,N); action (B) int64; value_new, value_old, adv, return_ (B);
 *             weight (B) or NULL; dual_clip <= 0 means None
 *             -> out5 = {policy_loss, value_loss, entropy_loss, approx_kl, clipfrac};
 *             saved: pol_coef (B) = dpolicy_loss/dlogp_new[a], val_coef (B) = dvalue_loss/dvalue_new
 *   backward: three upstream gradients (device scalars) -> grad_logits_new (B,N), grad_value_new (B) */
int hpc_rll_ppo_forward(const float* logits_new, const float* logits_old, const int64_t* action,
                        const float* value_new, const float* value_old, const float* adv, const float* return_,
                        const float* weight, float* out5, float* pol_coef, float* val_coef, int64_t B, int64_t N,
                        double clip_ratio, int use_value_clip, double dual_clip, int64_t global_B, void* workspace,
                        size_t workspace_bytes, void* stream);
/* same, with the advantage normalisation fused in: every sample uses (adv - adv_stats[0]) / adv_stats[1],
 * adv_stats = {mean, std + 1e-8} on the device as written by hpc_rll_adv_stats (origin/ppo.py:43-47 leaves
 * this step to the caller; doing it here saves a read+write of `adv`).  Backward is unchanged. */
int hpc_rll_ppo_forward_norm(const float* logits_new, const float* logits_old, const int64_t* action,
                             const float* value_new, const float* value_old, const float* adv, const float* return_,
                             const float* weight, const float* adv_stats, float* out5, float* pol_coef,
                             float* val_coef, int64_t B, int64_t N, double clip_ratio, int use_value_clip,
                             double dual_clip, int64_t global_B, void* workspace, size_t workspace_bytes,
                             void* stream);
int hpc_rll_ppo_backward(const float* grad_policy_loss, const float* grad_value_loss, const float* grad_entropy_loss,
                         const float* logits_new, const int64_t* action, const float* weight, const float* pol_coef,
                         const float* val_coef, float* grad_logits_new, float* grad_value_new, int64_t B, int64_t N,
                         int64_t global_B, void* stream);

/* ---- n-step TD-error family ------------------------------------------------------------------
 * Common: reward (T,B) with T = nstep; done (B) as FLOAT 0/1 (the reference reads it as float*,
 * src/rl_utils/q_nstep_td.cu:39); weight (B) or NULL; action / next_n_action (B) int64.
 * Each forward returns loss[1], td_err (B) and grad_buf = d loss / d(gathered row) (no upstream grad);
 * each backward scatters g*grad_buf into the action's slot of a dense, otherwise zero gradient. */

/* q_nstep_td_error / q_nstep_td_error_with_rescale: replaces QNStepTd{,Rescale}{Forward,Backward}
 * (/root/reference/src/rl_utils/q_nstep_td.cu, q_nstep_td_rescale.cu; kernels q_nstep_td_kernel.h:11-62,
 * q_nstep_td_rescale_kernel.h:11-72); semantics hpc_rll/origin/td.py:252-291, 294-340.
 *   q, next_n_q (B,N); grad_buf (B); grad_q (B,N) */
int hpc_rll_q_nstep_td_forward(const float* q, const float* next_n_q, const int64_t* action,
                               const int64_t* next_n_action, const float* reward, const float* done,
                               const float* weight, float* loss, float* td_err, float* grad_buf, int64_t T,
                               int64_t B, int64_t N, double gamma, int rescale, int64_t global_B, void* workspace,
                               size_t workspace_bytes, void* stream);
int hpc_rll_q_nstep_td_backward(const float* grad_loss, const float* grad_buf, const int64_t* action,
                                float* grad_q, int64_t B, int64_t N, void* stream);

/* dist_nstep_td_error (C51): replaces DistNStepTd{Forward,Backward} (/root/reference/src/rl_utils/
 * dist_nstep_td.cu:8-98, kernels dist_nstep_td_kernel.h:11-107); semantics hpc_rll/origin/td.py:29-143.
 *   dist, next_n_dist (B,N,n_atom); grad_buf (B,n_atom); grad_dist (B,N,n_atom) */
int hpc_rll_dist_nstep_td_forward(const float* dist, const float* next_n_dist, const int64_t* action,
                                  const int64_t* next_n_action, const float* reward, const float* done,
                                  const float* weight, float* loss, float* td_err, float* grad_buf, int64_t T,
                                  int64_t B, int64_t N, int64_t n_atom, double gamma, double v_min, double v_max,
                                  int64_t global_B, void* workspace, size_t workspace_bytes, void* stream);
int hpc_rll_dist_nstep_td_backward(const float* grad_loss, const float* grad_buf, const int64_t* action,
                                   float* grad_dist, int64_t B, int64_t N, int64_t n_atom, void* stream);

/* qrdqn_nstep_td_error: replaces QRDQNNStepTDError{Forward,Backward} (/root/reference/src/rl_utils/
 * qrdqn_nstep_td_error.cu:8-95, kernels qrdqn_nstep_td_error_kernel.h:11-106); semantics
 * hpc_rll/origin/td.py:455-517 with `tau` the INTEGER quantile count (as the reference wrapper passes it).
 *   q, next_n_q (B,N,tau); value_gamma (B) or NULL (= gamma^T); grad_buf (B,tau); grad_q (B,N,tau) */
int hpc_rll_qrdqn_nstep_td_forward(const float* q, const float* next_n_q, const int64_t* action,
                                   const int64_t* next_n_action, const float* reward, const float* done,
                                   const float* weight, const float* value_gamma, float* loss, float* td_err,
                                   float* grad_buf, int64_t tau, int64_t T, int64_t B, int64_t N, double gamma,
                                   int64_t global_B, void* workspace, size_t workspace_bytes, void* stream);
int hpc_rll_qrdqn_nstep_td_backward(const float* grad_loss, const float* grad_buf, const int64_t* action,
                                    float* grad_q, int64_t tau, int64_t B, int64_t N, void* stream);

/* iqn_nstep_td_error: replaces IQNNStepTDError{Forward,Backward} (/root/reference/src/rl_utils/
 * iqn_nstep_td_error.cu:8-100, kernels iqn_nstep_td_error_kernel.h:11-108); semantics
 * hpc_rll/origin/td.py:361-448.
 *   q (tau,B,N); next_n_q (tau',B,N); replay_quantiles (tau,B); grad_buf (tau,B); grad_q (tau,B,N) */
int hpc_rll_iqn_nstep_td_forward(const float* q, const float* next_n_q, const int64_t* action,
                                 const int64_t* next_n_action, const float* reward, const float* done,
                                 const float* replay_quantiles, const float* weight, const float* value_gamma,
                                 float* loss, float* td_err, float* grad_buf, int64_t tau, int64_t tau_prime,
                                 int64_t T, int64_t B, int64_t N, double gamma, double kappa, int64_t global_B,
                                 void* workspace, size_t workspace_bytes, void* stream);
int hpc_rll_iqn_nstep_td_backward(const float* grad_loss, const float* grad_buf, const int64_t* action,
                                  float* grad_q, int64_t tau, int64_t B, int64_t N, void* stream);

/* ---- the path's only collective: all-reduce(SUM) of <= 16 loss scalars over NVLink peer memory -------------------
 * Batch-sharded loss ops (kernels normalise by `global_B`) end in a sum of a few scalars over the ranks.  Instead of an NCCL
 * call, every rank owns a small device buffer its peers have mapped through CUDA IPC; one tiny kernel per rank stores
 * its epoch-tagged scalars into every peer's buffer, waits for all ranks' words in its own buffer and adds them in RANK
 * ORDER (bit-identical on every rank, run to run).  Set-up (once per process group):
 *   hpc_rll_p2p_alloc  -> local buffer + 64-byte IPC handle; exchange the handles (e.g. torch.distributed.all_gather);
 *   hpc_rll_p2p_open   -> a mapping of each peer's buffer;  bufs[r] = peer mapping, bufs[rank] = the local buffer.
 * hpc_rll_allreduce_scalars_p2p reduces vals[0..n) (device, fp32) in place on `stream`; every rank must issue the same
 * sequence of calls.  Capturable in CUDA graphs (the epoch lives on the device).  di_hpc_b200/sharding.py wraps it. */
size_t hpc_rll_p2p_buffer_bytes(void);
int hpc_rll_p2p_alloc(void** local_buf, void* ipc_handle_64);
int hpc_rll_p2p_open(const void* ipc_handle_64, void** peer_buf);
int hpc_rll_p2p_close(void* peer_buf);
int hpc_rll_p2p_free(void* local_buf);
int hpc_rll_allreduce_scalars_p2p(float* vals, int n, void* const* bufs, int rank, int world, void* stream);

/* ---- ragged-tensor padding (the data format on the input side of the path) -----------------------
 * replaces Pad{1,2,3}DForward / GroupPad{1,2,3}DForward / Unpad{1,2,3}DForward and the two group splitters
 * (/root/reference/src/rl_utils/padding.cu:8-589, kernels include/hpc/rll/cuda/rl_utils/padding_kernel.h:100-233);
 * semantics of hpc_rll/origin/padding.py.  Descriptor tables are HOST arrays of length n (device pointers
 * inside); shapes / padded are n x 3 int32, right-aligned (leading dims 1 for 1-D / 2-D).  No allocation, no copy: the
 * tables ride in kernel parameter space.
 *   pad  : dst[k] (padded slot, prod(padded[k]) floats) = src[k] inside shapes[k], `value` elsewhere;
 *          mask[k] (int32) = 1 inside, `value` elsewhere
 *   unpad: dst[k] (prod(shapes[k]) floats) = the leading shapes[k] block of the padded slot src[k] */
int hpc_rll_pad_batch(const float* const* src, float* const* dst, int32_t* const* mask, const int32_t* shapes,
                      const int32_t* padded, int64_t n, int value, void* stream);
int hpc_rll_unpad_batch(const float* const* src, float* const* dst, const int32_t* shapes, const int32_t* padded,
                        int64_t n, void* stream);
/* host-only helpers: split a size-sorted shape list (n x ndim int64) into groups.
 * oracle: exactly `group` groups minimising the padded volume; positions[0..group], positions[group] = n.
 * sample: random boundaries (deterministic per seed), equal-shaped neighbours merged; starts[0..*n_groups]. */
int hpc_rll_oracle_split_group(const int64_t* shapes, int64_t n, int ndim, int group, int64_t* positions);
int hpc_rll_sample_split_group(const int64_t* shapes, int64_t n, int ndim, int group, uint64_t seed,
                               int64_t* starts, int* n_groups);

/* ---- ScatterConnection (AlphaStar-style entity -> spatial map scatter) ----------------------------
 * replaces ScatterConnectionForward / ScatterConnectionBackward of the reference's `hpc_torch_utils_network`
 * (/root/reference/src/torch_utils/network/scatter_connection.cu:8-76, kernels
 * include/hpc/rll/cuda/torch_utils/network/scatter_connection_kernel.h:60-120); semantics of
 * hpc_rll/origin/scatter_connection.py:25-64 on the CPU, i.e. sequential in entity order m.
 *   forward : x (B,M,N), location (B,M,2) int64 pairs (y, x) -> out (B,N,H,W), every element written once:
 *             mode 1 (add)   out[b,n,y*W+x] = ((0.f + x[b,m0,n]) + x[b,m1,n]) + ... in ascending m
 *             mode 0 (cover) out[b,n,y*W+x] = x[b,m_last,n] (the last entity at a cell wins)
 *             cells no entity lands on are +0.f; no memset is needed before the call
 *   backward: grad_out (B,N,H,W) -> grad_x (B,M,N), grad_x[b,m,n] = grad_out[b,n,y*W+x] (both modes)
 * An entity with y outside [0,H) or x outside [0,W) writes nothing and gets a zero gradient.  No atomics:
 * results are bit-identical run to run.  No workspace.  Contiguous tensors; any 4-byte alignment. */
int hpc_rll_scatter_connection_forward(const float* x, const int64_t* location, float* out, int64_t B, int64_t M,
                                       int64_t N, int64_t H, int64_t W, int mode /* 0 cover, 1 add */, void* stream);
int hpc_rll_scatter_connection_backward(const float* grad_out, const int64_t* location, float* grad_x, int64_t B,
                                        int64_t M, int64_t N, int64_t H, int64_t W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HPC_RLL_B200_H_ */
