// Kernel argument blocks and launcher prototypes (internal to libtcelbo.so).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "tc_layout.h"
#include "tc_common.cuh"

namespace tcelbo {

struct FwdArgs {
    const float* zs; const float* ns; const float* qmax;   // [bl_pad][dp]
    const float* mu_pad;                                   // [bg_pad][dp]
    float* s2; int64_t ld_s2;                              // joint exponents (nullptr: not saved)
    float* Spart;                                          // [n_js][bl_pad][dp]
    float* Jpart;                                          // [n_js][bl_pad] (m, s) pairs
    int b_loc, bl_pad, bg_pad, row_offset, js_len;
    Segments seg; int n_rb;                                // balanced segments (row-variance sweep; tc_layout.h: plan_segments)
    Weights w;
};

struct FinArgs {
    const float* Spart; const float* Jpart; const float* shift;
    float* S; float* J2; float* log_qz; float* log_qz_prod;
    int b_loc, bl_pad, d, dp, n_js;
    Segments seg; int tiles_per_block, rows_per_block;     // seg.n_ctas > 0: per-row slot count from the segment plan instead of n_js
    float lw_u;
    // optional fusion of solvers/tc.py:83-89: kl_i (ops.py:161-163) and loss_i = (beta-1)*(log_qz-log_qz_prod) + kl_i
    const float* lv; int64_t ldlv; const float* mu_loc; int64_t ldmu;   // this rank's rows of logvar / mu (nullptr: no fusion)
    float beta; float* loss_rows; float* kl_rows;
    // optional batch-level epilogue, reduced deterministically by the last CTA to finish (fixed summation order):
    //   loss_mean = mean_i loss_rows[i], kl_mean = mean_i kl_rows[i]               (solvers/tc.py:83-89 with reduce="mean")
    //   e_rows[i] = exp(-2*scale*(rec_rows[i] + loss_rows[i])), expelbo = mean_i e_rows[i]   (solvers/intro.py:102-103)
    float* loss_mean; float* kl_mean; const float* rec_rows; float scale; float* expelbo; float* e_rows;
    float* red_part; unsigned int* ticket;                       // [3][gridDim.x] partial sums, arrival counter (zeroed by the prologue)
};

// One prologue kernel: pads / gathers the column operand, derives the per-(i,d) row constants, optionally forms
// z = mu + eps * exp(logvar / 2) on the fly (ops.py:183-185), zeroes the finalize kernel's ticket.
struct PrepArgs {
    const float* mu_all; int64_t ldmu;                           // [b_glob][d] columns (ignored when parts != nullptr)
    const float* const* parts; int64_t ld_part; int rows_per_part;   // peer exchange: one [rows_per_part][d] block per rank
    const float* z; int64_t ldz;                                 // sampled latents of the local rows, or nullptr with eps set
    const float* eps; int64_t ldeps; const float* mu_loc; int64_t ldmu_loc; float* z_out; int64_t ldz_out;
    const float* logvar; int64_t ldlv;
    int b_loc, b_glob, d, bl_pad, bg_pad, dp;
    float* mu_pad; float* zs; float* ns; float* qmax; float* shift; float* vr;
    unsigned int* ticket;
    PeerSync sync;                                               // peer exchange: barrier between the ranks' publish and this gather
};

struct BwdFusedArgs {
    const float* zs; const float* ns; const float* qmax; const float* gps;   // [bl_pad][dp]
    const float* gj; const float* J2;                                        // [bl_pad]
    const float* mu_pad;                                                     // [bg_pad][dp]
    const float* s2; int64_t ld_s2;
    float* Apart; float* CRpart;                                             // [n_js][bl_pad][dp]
    float* Gacc;                                                             // [bg_pad][dp], zeroed by the caller
    float* Gacc2;                                                            // column-variance variant: logvar column sums
    int b_loc, bl_pad, bg_pad, row_offset, js_len;
    int pitch;                                                               // floats per row of the [*, dp] arrays
    Segments seg; int n_blocks, n_rb;                                        // balanced segments (fused sweep; tc_layout.h: plan_segments)
    int plan_only;                                                           // host-side: compute the column split, launch nothing
    Weights w;
};

struct BwdFinArgs {
    const float* Apart; const float* CRpart; const float* Gpart;
    const float* ns; const float* vr;
    float* grad_z; int64_t ldgz; float* grad_lv; int64_t ldglv; float* grad_mu; int64_t ldgmu;
    int b_loc, b_glob, bl_pad, bg_pad, d, dp, n_js, n_is;
    // fused sweep: the partial slots of a row come from the segments that touch its (slice, row block) block
    Segments seg; int tiles_per_block, n_rb, rows_per_block, slice_dp;
    // optional fused KL gradient (ops.py:161-163): gk_i * mu on this rank's rows of grad_mu, gk_i * 0.5*(exp(lv)-1) on grad_lv
    const float* gk; const float* lv; int64_t ldlv; const float* mu_all; int64_t ldmu; int row_offset;
    // peer-memory exchange: every rank's backward scratch (device table of n_ranks base pointers); the column sums of this
    // rank's rows are read straight from the peers' accumulators and grad_mu covers the local rows only (nullptr: grad_mu_all)
    const void* const* scratch_parts; size_t g_off; int n_ranks;
    // fused reparameterize backward (ops.py:183-185): with eps set, the local rows of grad_mu also receive grad_z and grad_lv
    // receives grad_z * eps * 0.5 * exp(logvar / 2), i.e. the outputs are the gradients w.r.t. the encoder's mu / logvar
    const float* eps; int64_t ldeps;
    PeerSync sync;                                               // peer exchange: barrier between the ranks' sweeps and this reduce
};

cudaError_t launch_prep(const PrepArgs& a, cudaStream_t st);
cudaError_t launch_publish(const float* src, int64_t ld, int b_loc, int d, float* dst, unsigned int* epoch, cudaStream_t st);
cudaError_t launch_fwd(const Plan& p, const FwdArgs& a, cudaStream_t st);
cudaError_t launch_fwd_finalize(const Plan& p, const FinArgs& a, cudaStream_t st);
// Upstream gradients of the backward prologue.  Per row i (any pointer may be null):
//   gl_i = g_loss[i] + g_loss_mean[0]/b_loc + g_expelbo[0] * (-2*scale/b_loc) * e_rows[i]      (dLoss/dloss_rows[i])
//   gJ_i = g_log_qz[i] + (beta-1)*gl_i,  gP_i = g_log_qz_prod[i] - (beta-1)*gl_i,  gk_i = gl_i + g_kl[i] + g_kl_mean[0]/b_loc
// The prologue writes gps = gP/S, gj = gJ, gk (if gk != null), g_rec_rows[i] = the exp-ELBO part of gl_i (the gradient of
// rec_rows, if asked for) and zeroes `zero_n` floats at `zero` (the column accumulator).
struct BwdUpstream {
    const float* g_log_qz; const float* g_log_qz_prod; const float* g_loss; const float* g_kl;
    const float* g_loss_mean; const float* g_kl_mean; const float* g_expelbo; const float* e_rows; float scale;
    float* g_rec_rows;
    float beta;
    unsigned int* epoch;          // peer exchange with in-kernel barriers: the backward barrier counter this prologue advances
};
cudaError_t launch_bwd_prep(const Plan& p, const BwdUpstream& u, const float* S, float* gps, float* gj, float* gk,
                            float* zero, size_t zero_n, cudaStream_t st);
cudaError_t launch_bwd_fused(const Plan& p, const BwdFusedArgs& a, BwdFinArgs* fin, cudaStream_t st);   // fills fin's segment fields
// column-variance ("full" path) variant, tc_colvar.cu
cudaError_t launch_colvar_prep(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* lv_all, int64_t ldlv,
                               const Plan& p, float* colpack, float* zpad, float* shift, cudaStream_t st);
cudaError_t launch_fwd_colvar(const Plan& p, const FwdArgs& a, int* n_js_out, cudaStream_t st);
cudaError_t launch_bwd_colvar(const Plan& p, const BwdFusedArgs& a, int* n_js_out, cudaStream_t st);
cudaError_t launch_bwd_colvar_finalize(const Plan& p, const BwdFinArgs& a, const float* colpack, const float* Glv, cudaStream_t st);
cudaError_t launch_bwd_fused_finalize(const Plan& p, const BwdFinArgs& a, cudaStream_t st);

}  // namespace tcelbo
