/*
 * tcelbo.h -- C ABI of the B200-native total-correlation ELBO path (libtcelbo.so).
 *
 * Drop-in boundary for the hot path of meffmadd/intro-tc-vae (file:line relative to the reference
 * repository).  The reference is pure Python/PyTorch with no FFI of its own; these entry points are
 * what a binding for the path would bind, one per reference function:
 *
 *   tcelbo_forward / tcelbo_backward    ops.py:52-89   total_correlation
 *                                       ops.py:15-21   gaussian_log_density_torch   (TCELBO_VAR_ROW)
 *                                       ops.py:24-29   gaussian_log_density         (TCELBO_VAR_COL,
 *                                                      as called at solvers/tc.py:114-116)
 *                                       ops.py:32-49   log_importance_weight_matrix (folded in: 3 scalars)
 *                                       ops.py:104-115 minibatch_stratified_sampling (TCELBO_EST_MSS)
 *                                       ops.py:92-101  minibatch_weighted_sampling   (TCELBO_EST_MWS)
 *   tcelbo_kl_forward / _backward       ops.py:136-163 kl_divergence / kl_no_reduce
 *   tcelbo_reparam_forward / _backward  ops.py:166-185 reparameterize (eps supplied by the caller so
 *                                                      that torch's device Philox stream is preserved)
 *   tcelbo_rowdensity_forward/_backward ops.py:24-29 summed over dim 1, the row-wise log q(z|x) and
 *                                       log p(z) terms of solvers/tc.py:107,112
 *
 * Conventions
 *   - All pointers are DEVICE pointers to fp32 unless stated; `ld*` are row pitches in ELEMENTS
 *     (the encoder returns mu/logvar as chunk views with pitch 2*D, models.py:242-244).
 *   - Nothing is allocated, no host synchronisation happens, every call is asynchronous on `stream`
 *     (a cudaStream_t passed as void*) and CUDA-graph capturable.  Scratch comes from the caller:
 *     query tcelbo_workspace_bytes() and pass a 256-byte aligned buffer.  The buffer written by
 *     tcelbo_forward(flags | TCELBO_SAVE_FOR_BACKWARD) must be handed unchanged to tcelbo_backward,
 *     which only reads it and writes its own scratch (tcelbo_backward_scratch_bytes()).
 *   - Return value: 0 on success, a TCELBO_ERR_* code otherwise; tcelbo_last_error() returns a
 *     thread-local message.  Nothing throws across the boundary.
 *   - Sharding (SURVEY.md 8e): a rank owns global rows [row_offset, row_offset + b_loc) of a global
 *     batch of b_glob columns; `mu_all` (and `logvar` for TCELBO_VAR_COL) hold all b_glob rows after
 *     the caller's all-gather; grad_mu_all is this rank's partial [b_glob, D] to be reduce-scattered.
 *     Single GPU: b_loc == b_glob, row_offset == 0.
 *   - Error behaviour mirrored from the reference: b_glob == 1 is rejected (ZeroDivisionError at
 *     ops.py:44, raised by the Python wrapper); dataset_size < b_glob-1 yields NaN outputs (log of a
 *     negative weight), not an error.
 */
#ifndef TCELBO_H_
#define TCELBO_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCELBO_VERSION 3

/* flags */
#define TCELBO_EST_MSS            0u   /* minibatch stratified sampling (active in the reference) */
#define TCELBO_EST_MWS            1u   /* minibatch weighted sampling */
#define TCELBO_VAR_ROW            0u   /* log q(z_i | mu_j, var_i), variance floored at 1e-4 (ops.py:15-21,80-82) */
#define TCELBO_VAR_COL            2u   /* log q(z_i | mu_j, var_j), no floor (ops.py:24-29, solvers/tc.py:114-116) */
#define TCELBO_SAVE_FOR_BACKWARD  4u   /* forward keeps what backward needs in the workspace */

/* error codes */
#define TCELBO_OK               0
#define TCELBO_ERR_INVALID      1      /* bad argument (message says which) */
#define TCELBO_ERR_CUDA         2      /* a CUDA runtime call failed */
#define TCELBO_ERR_WORKSPACE    3      /* workspace too small or misaligned */
#define TCELBO_ERR_UNSUPPORTED  4      /* shape outside the built kernels (D > 512) */

int         tcelbo_version(void);
const char* tcelbo_last_error(void);

/* Bytes of the forward workspace (larger with TCELBO_SAVE_FOR_BACKWARD: it then keeps the per-row results and
 * the b_loc x b_glob joint exponents that backward reads; never the b x b x d log-densities). */
size_t tcelbo_workspace_bytes(int b_loc, int b_glob, int d, uint32_t flags);
/* Bytes of the separate scratch buffer tcelbo_backward writes (the forward workspace is read-only there). */
size_t tcelbo_backward_scratch_bytes(int b_loc, int b_glob, int d, uint32_t flags);

/*
 * Forward: for each local row i
 *   log_qz_prod[i] = sum_d LSE_j( logw_ij + lp_ijd )        (log prod_d q(z_d))
 *   log_qz[i]      =       LSE_j( logw_ij + sum_d lp_ijd )   (log q(z))
 * total correlation is log_qz - log_qz_prod (ops.py:86-89).
 *   z       [b_loc , D]  sampled latents of the local rows
 *   mu_all  [b_glob, D]  encoder means of ALL rows (columns j)
 *   logvar  [b_loc , D]  for TCELBO_VAR_ROW (local rows); [b_glob, D] for TCELBO_VAR_COL
 */
int tcelbo_forward(const float* z, int64_t ldz,
                   const float* mu_all, int64_t ldmu,
                   const float* logvar, int64_t ldlv,
                   int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                   float* log_qz, float* log_qz_prod,
                   void* workspace, size_t workspace_bytes, void* stream);

/*
 * Backward of tcelbo_forward given g_log_qz[i] = dLoss/dlog_qz[i], g_log_qz_prod[i] likewise.
 * The B x B x D log-densities are recomputed tile by tile, never stored.
 *   grad_z       [b_loc , D]
 *   grad_mu_all  [b_glob, D]  (partial over this rank's rows)
 *   grad_logvar  [b_loc , D] for TCELBO_VAR_ROW, [b_glob, D] (partial) for TCELBO_VAR_COL
 * Same z / mu_all / logvar / sizes / flags as the forward call whose workspace is passed.
 */
int tcelbo_backward(const float* z, int64_t ldz,
                    const float* mu_all, int64_t ldmu,
                    const float* logvar, int64_t ldlv,
                    int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                    const float* g_log_qz, const float* g_log_qz_prod,
                    float* grad_z, int64_t ldgz,
                    float* grad_mu_all, int64_t ldgmu,
                    float* grad_logvar, int64_t ldglv,
                    const void* workspace, size_t workspace_bytes,
                    void* scratch, size_t scratch_bytes, void* stream);

/*
 * Fused compute_kl_loss of TCSovler._compute_kl_loss_simple (solvers/tc.py:69-89), row-variance density:
 *   kl_rows[i]   = -0.5 * sum_d (1 + logvar - exp(logvar) - mu^2)                      (ops.py:161-163)
 *   loss_rows[i] = (beta - 1) * (log_qz[i] - log_qz_prod[i]) + kl_rows[i]
 * Same arguments as tcelbo_forward / tcelbo_backward; mu of this rank's rows is read from
 * mu_all[row_offset .. row_offset + b_loc).  The backward takes dLoss/dloss_rows (required) and optionally
 * dLoss/dkl_rows, dLoss/dlog_qz, dLoss/dlog_qz_prod (NULL = zero); the KL gradient is added to grad_logvar and to
 * this rank's rows of grad_mu_all, so no separate KL kernels or elementwise combine kernels are launched.
 */
int tcelbo_klloss_forward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                          int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                          float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod,
                          void* workspace, size_t workspace_bytes, void* stream);
int tcelbo_klloss_backward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                           int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                           const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                           float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                           const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream);

/*
 * Optional fusions around the fused loss (SURVEY.md 8f rank 1); a NULL member switches its fusion off, a NULL struct all of them.
 *   prologue  reparameterize, ops.py:183-185: with `eps` set, z is NOT read (pass NULL); z = mu + eps * exp(logvar / 2) of this
 *             rank's rows is formed inside the prologue kernel and, if z_out != NULL, stored there for the decoder.  The
 *             backward (same `eps`) then applies the chain rule through z itself: grad_logvar and this rank's rows of
 *             grad_mu_all are the gradients w.r.t. the ENCODER outputs; grad_z still receives dLoss/dz.
 *   epilogue  batch means, solvers/tc.py:83-89 with reduce="mean": loss_mean[0] = mean_i loss_rows[i], kl_mean[0] likewise
 *             (mean over this rank's b_loc rows, summed in a fixed order);
 *             soft-intro exp-ELBO term, solvers/intro.py:102-103 with kl_i = loss_rows[i] (solvers/intro.py:84-89):
 *             e_rows[i] = exp(-2 * scale * (rec_rows[i] + loss_rows[i])), expelbo[0] = mean_i e_rows[i].
 *   backward  g_loss_mean / g_kl_mean / g_expelbo are DEVICE scalars (dLoss/d of the three means); e_rows is the forward's;
 *             g_rec_rows [b_loc] (optional output) receives dLoss/drec_rows[i] = g_expelbo * (-2 scale / b_loc) * e_rows[i].
 */
typedef struct tcelbo_fusion {
    const float* eps; int64_t ldeps;
    float* z_out; int64_t ldz_out;
    float* loss_mean; float* kl_mean;
    const float* rec_rows; float scale; float* expelbo; float* e_rows;
    const float* g_loss_mean; const float* g_kl_mean; const float* g_expelbo; float* g_rec_rows;
} tcelbo_fusion;

/* tcelbo_klloss_forward / _backward with the fusions above; every per-row upstream gradient of the backward may be NULL as long
 * as one upstream gradient (per-row or scalar) is given. */
int tcelbo_klloss_forward_ex(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                             int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                             float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod, const tcelbo_fusion* fusion,
                             void* workspace, size_t workspace_bytes, void* stream);
int tcelbo_klloss_backward_ex(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                              int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                              const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                              const tcelbo_fusion* fusion,
                              float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                              const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream);

/*
 * Peer-memory exchange for the row-sharded fused loss (one process per GPU; SURVEY.md 8e).  Replaces the NCCL all-gather of
 * the column operand and the reduce-scatter of its gradient (what a torch DistributedDataParallel port of solvers/tc.py:69-89
 * would issue around ops.py:52-89) by loads over NVLink inside the library's own prep / finalize kernels:
 *   forward : every rank publishes its [b_loc, d] rows of mu in a buffer that is mapped into all n_ranks processes (torch
 *             symmetric memory, cudaIpc, a VMM fabric handle ...); after a cross-rank barrier ON THE STREAM (the caller's), the
 *             column-prep kernel gathers the rows of all ranks through `mu_parts`, a DEVICE array of n_ranks pointers
 *             (entry p = rank p's rows, row pitch ld_part floats).  b_glob = n_ranks * b_loc, row_offset = rank * b_loc.
 *   backward: `scratch` must itself live in such a mapped buffer.  TCELBO_PEER_SWEEP runs the gradient sweep and leaves the
 *             column sums in this rank's scratch; after another barrier, TCELBO_PEER_FINISH sums this rank's rows over the
 *             scratch buffers of all ranks (`scratch_parts`, DEVICE array of n_ranks scratch base pointers) and writes
 *             grad_z, grad_logvar and grad_mu_loc [b_loc, d] (the already reduce-scattered gradient of mu, KL term included).
 * A scratch (and a published mu buffer) may be reused two exchanges later (double-buffer them), never by the very next one.
 * `mu_loc` is this rank's rows of mu (the KL term reads it).  Row-variance density only.  `fusion` as in the _ex entry points
 * (NULL = none): with `eps`, z is formed in the prologue and grad_mu_loc / grad_logvar are the gradients w.r.t. the encoder outputs.
 */
/* Optional in-kernel barriers for the two exchange steps (NULL: the CALLER puts a cross-rank barrier on the stream before
 * tcelbo_klloss_forward_peer and before the TCELBO_PEER_FINISH call, as described above).  With it, the prologue kernel signals
 * "my rows are published" to every rank and waits for all ranks before it gathers (its row work overlaps the wait), and the
 * finalize kernel does the same for "my sweep is done" before it reduces: no barrier launches at all.  Every rank must then
 * issue the same sequence of peer calls; a rank that never arrives makes the others trap after ~30 s.
 *   flag_parts  DEVICE table of n_ranks pointers; entry r = rank r's flag array of 2*n_ranks 32-bit words, zero-initialised
 *               once (before the first call, with a real barrier after the zeroing), mapped into every process
 *   state       DEVICE, local to this rank: 4 zero-initialised 32-bit words (the barrier counters of the two exchanges)
 * The counters are advanced by the kernel BEFORE the waiting one on the stream: tcelbo_peer_publish (which also copies this
 * rank's rows of mu into its mapped buffer) for the forward exchange -- call it instead of a plain copy -- and the backward
 * prologue (TCELBO_PEER_SWEEP) for the backward exchange. */
typedef struct tcelbo_peer_sync {
    unsigned int* const* flag_parts;
    unsigned int* state;
} tcelbo_peer_sync;

int tcelbo_peer_publish(const float* mu_loc, int64_t ldmu, int b_loc, int d, float* published /* [b_loc, d] dense, mapped */,
                        const tcelbo_peer_sync* sync, void* stream);

#define TCELBO_PEER_SWEEP  1
#define TCELBO_PEER_FINISH 2
int tcelbo_klloss_forward_peer(const float* z, int64_t ldz, const float* mu_loc, int64_t ldmu,
                               const float* const* mu_parts, int64_t ld_part, const float* logvar, int64_t ldlv,
                               int b_loc, int n_ranks, int rank, int d, int64_t dataset_size, uint32_t flags, float beta,
                               float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod,
                               const tcelbo_fusion* fusion, const tcelbo_peer_sync* sync,
                               void* workspace, size_t workspace_bytes, void* stream);
int tcelbo_klloss_backward_peer(int phase, const float* z, int64_t ldz, const float* mu_loc, int64_t ldmu,
                                const float* logvar, int64_t ldlv, int b_loc, int n_ranks, int rank, int d,
                                int64_t dataset_size, uint32_t flags, float beta,
                                const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                                float* grad_z, int64_t ldgz, float* grad_mu_loc, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                                const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                                const void* const* scratch_parts, const tcelbo_fusion* fusion, const tcelbo_peer_sync* sync,
                                void* stream);

/* kl_rows[i] = -0.5 * sum_d (1 + logvar - exp(logvar) - mu^2)   (ops.py:161-163; argument order logvar, mu) */
int tcelbo_kl_forward(const float* logvar, int64_t ldlv, const float* mu, int64_t ldmu,
                      int b, int d, float* kl_rows, void* stream);
/* grad_logvar = g_rows[i] * 0.5*(exp(logvar)-1), grad_mu = g_rows[i] * mu */
int tcelbo_kl_backward(const float* logvar, int64_t ldlv, const float* mu, int64_t ldmu,
                       const float* g_rows, int b, int d,
                       float* grad_logvar, int64_t ldglv, float* grad_mu, int64_t ldgmu, void* stream);

/* z = mu + eps * exp(0.5*logvar)   (ops.py:183-185) */
int tcelbo_reparam_forward(const float* mu, int64_t ldmu, const float* logvar, int64_t ldlv,
                           const float* eps, int64_t ldeps, int b, int d, float* z, int64_t ldz, void* stream);
/* grad_mu = g_z ; grad_logvar = g_z * eps * 0.5*exp(0.5*logvar) */
int tcelbo_reparam_backward(const float* logvar, int64_t ldlv, const float* eps, int64_t ldeps,
                            const float* g_z, int64_t ldgz, int b, int d,
                            float* grad_mu, int64_t ldgmu, float* grad_logvar, int64_t ldglv, void* stream);
/* same, added to grad_mu / grad_logvar (which already hold the gradients of the loss terms that read mu and logvar directly) */
int tcelbo_reparam_backward_acc(const float* logvar, int64_t ldlv, const float* eps, int64_t ldeps,
                                const float* g_z, int64_t ldgz, int b, int d,
                                float* grad_mu, int64_t ldgmu, float* grad_logvar, int64_t ldglv, void* stream);

/*
 * Row-wise Gaussian log-density summed over D (ops.py:24-29 + .sum(dim=1), solvers/tc.py:107,112):
 *   out[i] = sum_d max(-0.5*((x-mu)^2*exp(-logvar) + logvar + log 2pi), -50)
 * mu == NULL and logvar == NULL mean the standard normal prior (zeros).
 */
int tcelbo_rowdensity_forward(const float* x, int64_t ldx, const float* mu, int64_t ldmu,
                              const float* logvar, int64_t ldlv, int b, int d, float* out, void* stream);
int tcelbo_rowdensity_backward(const float* x, int64_t ldx, const float* mu, int64_t ldmu,
                               const float* logvar, int64_t ldlv, const float* g_rows, int b, int d,
                               float* grad_x, int64_t ldgx, float* grad_mu, int64_t ldgmu,
                               float* grad_logvar, int64_t ldglv, void* stream);

/*
 * Callers either side of the path (SURVEY.md 8f):
 *   per-sample reconstruction loss, ops.py:188-236: out_rows[i] = sum over the n pixels of sample i of
 *     kind 0: (recon-x)^2   kind 1: |recon-x|   kind 2: binary cross entropy (logs clamped at -100);
 *     x and recon are contiguous [b, n]; `partial` is scratch of b * tcelbo_recloss_chunks(b, n) floats;
 *     the backward gives dLoss/drecon = g_rows[i] * d(elem)/d(recon) (x is detached in the reference).
 *   soft-intro exp-ELBO term, solvers/intro.py:102-103: out[0] = mean_i exp(-2*scale*(rec_rows[i] + kl_rows[i]));
 *     e_rows [b] is saved for the backward, which returns the common gradient of rec_rows and kl_rows.
 */
int tcelbo_recloss_chunks(int b, int64_t n);
int tcelbo_recloss_forward(const float* x, const float* recon, int b, int64_t n, int kind, float* partial, float* out_rows, void* stream);
int tcelbo_recloss_backward(const float* x, const float* recon, const float* g_rows, int b, int64_t n, int kind, float* grad_recon, void* stream);
int tcelbo_expelbo_forward(const float* rec_rows, const float* kl_rows, int b, float scale, float* out, float* e_rows, void* stream);
int tcelbo_expelbo_backward(const float* e_rows, const float* g_out, int b, float scale, float* g_rows, void* stream);

/*
 * Materialised-tensor helpers kept for API parity with the reference's ops.py (HBM-bound; the fused ops above never
 * build the tensor).  Densities: out[i,j,d] over a broadcast 3-D index space, operand strides in elements (0 on
 * broadcast dims); floored != 0 selects gaussian_log_density_torch (ops.py:15-21), else gaussian_log_density
 * (ops.py:24-29).  `shape`, `sx`, `sm`, `sl` are HOST arrays of three int64.  The backward writes elementwise
 * gradients at the broadcast shape (the caller reduces them over broadcast dims).
 */
int tcelbo_density_forward(int floored, const float* x, const float* mu, const float* logvar, const int64_t* shape,
                           const int64_t* sx, const int64_t* sm, const int64_t* sl, float* out, void* stream);
int tcelbo_density_backward(int floored, const float* x, const float* mu, const float* logvar, const float* g, const int64_t* shape,
                            const int64_t* sx, const int64_t* sm, const int64_t* sl, float* gx, float* gmu, float* glv, void* stream);
/* minibatch_stratified_sampling / minibatch_weighted_sampling (ops.py:104-115 / 92-101) on a contiguous [b,b,d] tensor;
 * lse_dim [b,d] and pair_sums [b,b] are saved for the backward. */
int tcelbo_sampling_forward(const float* log_qz_prob, int b, int d, int64_t dataset_size, uint32_t flags,
                            float* log_qz_prod, float* log_qz, float* lse_dim, float* pair_sums, void* stream);
int tcelbo_sampling_backward(const float* log_qz_prob, int b, int d, int64_t dataset_size, uint32_t flags,
                             const float* g_log_qz_prod, const float* g_log_qz, const float* lse_dim, const float* pair_sums,
                             const float* log_qz, float* grad_log_qz_prob, void* stream);

/* ---- diagnostics used by bench.py (no reference counterpart) --------------------------------------- */
/* Number of kernels this library has launched in the calling process so far. */
long long tcelbo_launch_count(void);
/* Bracket every later launch of one kernel class (1 = forward sweep, 2 = backward row sweep,
 * 3 = backward column sweep, 0 = off) with cudaEventRecord(start) / cudaEventRecord(stop) on its stream;
 * the events are cudaEvent_t handles owned by the caller.  Environment: TCELBO_PDL=0 launches the kernels without
 * programmatic dependent launch. */
int tcelbo_profile_events(int kernel_id, void* start_event, void* stop_event);
/* MUFU.EX2 saturation probe: `ctas` blocks of 256 threads, 8*iters dependent-chain ex2 per thread. */
int tcelbo_ex2_peak(float* scratch, int iters, int ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TCELBO_H_ */
