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
    Segments seg;                                          // balanced segments (row-variance sweep; tc_layout.h: plan_segments)
    int n_rb;                                              // read by no kernel, but dropping it moves `w` and with it changes the
    Weights w;                                             // register allocation (and spills) of the forward sweep kernels
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
    //   e_rows[i] = exp(-2*scale*(rec_rows[i] + loss_rows[i])), expelbo = mean_i e_rows[i]   (solvers/intro.py:102-103; with the
    //   loss_rows of either the fused KL loss or the decomposition)
    float* loss_mean; float* kl_mean; const float* rec_rows; float scale; float* expelbo; float* e_rows;
    // optional MI / TC / dimension-wise KL decomposition of solvers/tc.py:91-144 (column-variance plans; dz == nullptr: off),
    // per local row i with global row r = row_offset + i:
    //   condx_i = sum_d lp(z_id; mu_rd, lv_rd), pz_i = sum_d lp(z_id; 0, 0)      (lp: tc_common.cuh lp_unfloored, clamped)
    //   mi_i = condx_i - log_qz_i, tc_i = log_qz_i - log_qz_prod_i, dimkl_i = log_qz_prod_i - pz_i, loss_i = mi_i + beta*tc_i + dimkl_i
    //   dec_means[0..3] = the batch means of loss, mi, tc, dimkl (nullptr: none)
    // dz: the caller's z, or with the fused reparameterize the prologue's zero-padded z (the workspace's zpad, pitch dp)
    const float* dz; int64_t lddz; const float* dmu; int64_t lddmu; const float* dlv; int64_t lddlv;   // z rows; mu / logvar [b_glob]
    int row_offset;                                              // row of dmu / dlv holding local row 0 (0 with the peer exchange,
                                                                 // where dmu / dlv are this rank's rows only)
    float* dec_loss; float* dec_mi; float* dec_tc; float* dec_dimkl; float* dec_means;
    float* red_part; unsigned int* ticket;                       // [kFinRedSlots][gridDim.x] partial sums, arrival counter (zeroed by the prologue)
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

// Column-variance prologue (tc_colvar.cu): packs (sj, nmus, c2) of every column, zero-pads the local rows of z, optionally forming
// them as z = mu + eps * exp(logvar / 2) (ops.py:183-185).
struct ColPrepArgs {
    const float* z; int64_t ldz;                                 // this rank's rows, or nullptr with eps set
    const float* eps; int64_t ldeps; float* z_out; int64_t ldz_out;   // fused reparameterize (eps == nullptr: off; z_out optional)
    const float* mu_loc; const float* lv_loc;                    // this rank's rows of mu / logvar (pitches ldmu / ldlv), read with eps
    const float* mu_all; int64_t ldmu; const float* lv_all; int64_t ldlv;        // [b_glob][d] columns (ignored with parts)
    const float* const* mu_parts; const float* const* lv_parts; int64_t ld_part;  // peer exchange: one [b_loc][d] block per rank
    int b_loc, b_glob, d, bl_pad, bg_pad, dp;
    float* colpack; float* zpad; float* shift; unsigned int* ticket;
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
    // column-variance decomposition (BwdUpstream::gpz): the row-local gradients of condx_i (coefficient gc_i) and pz_i (gpz_i),
    // masked where lp < -50, on grad_z[i] and on row r = row_offset + i of grad_mu / grad_lv (nullptr: off).  With scratch_parts
    // (peer exchange) the column part covers rows [row_offset, row_offset + b_loc) only, sums the mu and logvar column sums of
    // every rank's scratch, and mu_all / lv / grad_mu / grad_lv are this rank's rows at local indices.  With eps, z is the
    // prologue's zpad (pitch dp) and the thread of (i, d) also writes row r of grad_mu / grad_lv, adding its own grad_z.
    const float* gc; const float* gpz; const float* z; int64_t ldz;
};

cudaError_t launch_prep(const PrepArgs& a, cudaStream_t st);
// src2 / dst2 (may be nullptr): a second [b_loc][d] block copied by the same kernel (logvar of the decomposition)
cudaError_t launch_publish(const float* src, int64_t ld, const float* src2, int64_t ld2, int b_loc, int d, float* dst, float* dst2,
                           unsigned int* epoch, cudaStream_t st);
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
    // MI / TC / dimension-wise KL decomposition (FinArgs::dz; gpz == nullptr: off).  g_loss / g_loss_mean carry the loss's
    // gradient as above, g_mi / g_tc / g_dimkl [b_loc] (any may be null) and g_dec_means[0..2] (the mi, tc, dimkl means; may be
    // null) the terms'; with gX_i = g_X[i] + g_dec_means[X]/b_loc:
    //   gJ_i = (beta-1)*gl_i - g_mi_i + g_tc_i,  gP_i = (1-beta)*gl_i - g_tc_i + g_dimkl_i,
    //   gk_i = gl_i + g_mi_i (coefficient of condx_i),  gpz[i] = -(gl_i + g_dimkl_i) (coefficient of pz_i)
    const float* g_mi; const float* g_tc; const float* g_dimkl; const float* g_dec_means; float* gpz;
};
cudaError_t launch_bwd_prep(const Plan& p, const BwdUpstream& u, const float* S, float* gps, float* gj, float* gk,
                            float* zero, size_t zero_n, cudaStream_t st);
cudaError_t launch_bwd_fused(const Plan& p, const BwdFusedArgs& a, cudaStream_t st);
// column-variance ("full" path) variant, tc_colvar.cu
cudaError_t launch_colvar_prep(const ColPrepArgs& a, cudaStream_t st);
cudaError_t launch_fwd_colvar(const Plan& p, const FwdArgs& a, cudaStream_t st);
cudaError_t launch_bwd_colvar(const Plan& p, const BwdFusedArgs& a, cudaStream_t st);
cudaError_t launch_bwd_colvar_finalize(const Plan& p, const BwdFinArgs& a, const float* colpack, const float* Glv, cudaStream_t st);
cudaError_t launch_bwd_fused_finalize(const Plan& p, const BwdFinArgs& a, cudaStream_t st);

}  // namespace tcelbo
