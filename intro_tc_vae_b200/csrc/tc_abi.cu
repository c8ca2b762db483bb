// C ABI of libtcelbo.so (include/tcelbo.h).  Plain pointers and sizes only; no torch types.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "tc_instr.h"
#include "tc_kernels.h"
#include "tc_materialized.h"
#include "tc_rowops.h"
#include "tcelbo.h"

using namespace tcelbo;

namespace tcelbo {
Instr& instr() { static Instr in; return in; }
}

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int fail_cuda(cudaError_t e, const char* what) {
    return fail(TCELBO_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

int sm_count() {
    static PerDevice cached_on;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) {
        int& cached = cached_on.cur();
        if (cached > 0) return cached;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) {
            cached = sms;
            return sms;
        }
    }
    (void)cudaGetLastError();
    return 148;                                   // B200; only reached when no device is visible (size queries on a CPU box)
}

// Importance weights the way the reference forms them (ops.py:42-49): python doubles rounded into an
// fp32 tensor, then log().  Only three distinct values exist, so the B x B matrix is never built.
Weights make_weights(int b_glob, int64_t n, uint32_t flags) {
    Weights w;
    w.b_glob = b_glob;
    if (flags & TCELBO_EST_MWS) {                 // ops.py:96,99: subtract log(B*N)
        w.mss = 0;
        w.r_n = w.r_s = 1.0f; w.l2r_n = w.l2r_s = 0.0f;
        w.lw_u = (float)(-std::log((double)b_glob * (double)n));
        return w;
    }
    const double m = (double)(b_glob - 1);
    const float w_u = (float)(1.0 / m);
    const float w_n = (float)(1.0 / (double)n);
    const float w_s = (float)(((double)n - m) / ((double)n * m));
    w.mss = 1;
    w.lw_u = logf(w_u);
    const double rn = (double)w_n / (double)w_u, rs = (double)w_s / (double)w_u;
    w.r_n = (float)rn;  w.l2r_n = (float)std::log2(rn);
    if (w_s < 0.0f) {                             // N < B-1: log of a negative weight is NaN in the reference
        w.r_s = NAN; w.l2r_s = NAN;
    } else {
        w.r_s = (float)rs; w.l2r_s = (float)std::log2(rs);    // rs == 0 -> -inf, rho 0: matches log(0) = -inf
    }
    return w;
}

bool aligned256(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 255u) == 0; }

template <typename T> T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

int check_common(const float* z, const float* mu_all, const float* logvar, int b_loc, int b_glob, int row_offset, int d,
                 int64_t dataset_size, uint32_t flags, int64_t ldz, int64_t ldmu, int64_t ldlv, bool z_optional = false) {
    if ((!z && !z_optional) || !mu_all || !logvar) return fail(TCELBO_ERR_INVALID, "null input pointer");
    if (b_loc < 1 || b_glob < 1 || d < 1) return fail(TCELBO_ERR_INVALID, "b_loc, b_glob and d must be positive");
    if (b_glob < 2 && !(flags & TCELBO_EST_MWS)) return fail(TCELBO_ERR_INVALID, "b_glob == 1: the stratified weight divides by B-1 (ZeroDivisionError at ops.py:44)");
    if (row_offset < 0 || (int64_t)row_offset + b_loc > b_glob) return fail(TCELBO_ERR_INVALID, "rows [row_offset, row_offset+b_loc) exceed b_glob");
    if (dataset_size < 1) return fail(TCELBO_ERR_INVALID, "dataset_size must be positive");
    if ((z && ldz < d) || ldmu < d || ldlv < d) return fail(TCELBO_ERR_INVALID, "row pitch smaller than d");
    if (d > 512) return fail(TCELBO_ERR_UNSUPPORTED, "d = %d > 512 is outside the built kernels", d);
    return TCELBO_OK;
}

}  // namespace

extern "C" {

int tcelbo_version(void) { return TCELBO_VERSION; }

const char* tcelbo_last_error(void) { return g_last_error.c_str(); }

size_t tcelbo_workspace_bytes(int b_loc, int b_glob, int d, uint32_t flags) {
    Plan p;
    if (!make_plan(p, b_loc, b_glob, d, flags, sm_count())) return 0;
    return p.total_bytes;
}

size_t tcelbo_backward_scratch_bytes(int b_loc, int b_glob, int d, uint32_t flags) {
    Plan p;
    if (!make_plan(p, b_loc, b_glob, d, flags, sm_count())) return 0;
    return p.bwd_bytes;
}

// ---- shared implementation of the plain and the loss-fused entry points ---------------------------------
struct LossFusion {            // solvers/tc.py:83-89 folded into the finalize kernels (null pointers: plain op)
    float beta = 1.0f;
    float* loss_rows = nullptr; float* kl_rows = nullptr;                 // forward outputs
    const float* g_loss = nullptr; const float* g_kl = nullptr;           // backward inputs
    bool on = false;
    tcelbo_fusion fz = {};                                                // optional prologue / epilogue fusions (tcelbo.h)
};

// Peer-memory exchange (tcelbo_*_peer): the column operand / the column accumulators live in n_ranks allocations that
// are all mapped into this process (NVLink peer memory); in that mode `mu_all` is this rank's rows only.
struct Peers {
    const float* const* mu_parts = nullptr; int64_t ld_part = 0;   // forward: device table of every rank's [b_loc, d] rows of mu
    const void* const* scratch_parts = nullptr;                    // backward finish: device table of every rank's scratch base
    int n_ranks = 0;
    int phase = 3;                                                 // backward: 1 = sweep into scratch, 2 = finish from the peers' scratch
    PeerSync sync = {nullptr, nullptr, 0, 0, 0};                   // in-kernel barrier (tcelbo_peer_sync) instead of the caller's
    bool on() const { return n_ranks > 0; }
};

static int forward_impl(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                        int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                        float* log_qz, float* log_qz_prod, const LossFusion& lf,
                        void* workspace, size_t workspace_bytes, void* stream, const Peers& peers = Peers()) {
    if (int rc = check_common(z, mu_all, logvar, b_loc, b_glob, row_offset, d, dataset_size, flags, ldz, ldmu, ldlv, lf.fz.eps != nullptr)) return rc;
    if (!log_qz || !log_qz_prod) return fail(TCELBO_ERR_INVALID, "null output pointer");
    if (lf.fz.eps && (lf.fz.ldeps < d || (lf.fz.z_out && lf.fz.ldz_out < d))) return fail(TCELBO_ERR_INVALID, "eps / z_out row pitch smaller than d");
    if (lf.fz.eps && (flags & TCELBO_VAR_COL)) return fail(TCELBO_ERR_UNSUPPORTED, "the fused reparameterize covers the row-variance density");
    if (lf.fz.expelbo && (!lf.fz.rec_rows || !lf.fz.e_rows)) return fail(TCELBO_ERR_INVALID, "expelbo needs rec_rows and e_rows");
    if (peers.on() && (flags & TCELBO_VAR_COL)) return fail(TCELBO_ERR_UNSUPPORTED, "the peer-memory exchange covers the row-variance density");
    Plan p;
    if (!make_plan(p, b_loc, b_glob, d, flags, sm_count())) return fail(TCELBO_ERR_INVALID, "cannot plan this shape");
    if (!workspace || workspace_bytes < p.total_bytes || !aligned256(workspace))
        return fail(TCELBO_ERR_WORKSPACE, "workspace must be 256-byte aligned and at least %zu bytes (got %zu)", p.total_bytes, workspace_bytes);
    if (lf.on && p.var_col) return fail(TCELBO_ERR_INVALID, "the fused (beta-1)*TC + KL loss uses the row-variance density (solvers/tc.py:69-89)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Weights w = make_weights(b_glob, dataset_size, flags);
    cudaError_t e;

    float* mu_pad = at<float>(workspace, p.off_mu);
    float* zs = at<float>(workspace, p.off_zs);
    float* ns = at<float>(workspace, p.off_ns);
    float* qmax = at<float>(workspace, p.off_qmax);
    float* shift = at<float>(workspace, p.off_shift);
    float* vr = at<float>(workspace, p.off_vr);
    float* Spart = at<float>(workspace, p.off_scratch);
    float* Jpart = Spart + (size_t)p.n_part_fwd * p.bl_pad * p.dp;

    const tcelbo_fusion& fz = lf.fz;
    unsigned int* ticket = at<unsigned int>(workspace, p.off_red) + 3 * (size_t)p.n_fin_ctas;
    if (p.var_col) {
        if ((e = launch_colvar_prep(z, ldz, mu_all, ldmu, logvar, ldlv, p, mu_pad, zs, shift, st)) != cudaSuccess) return fail_cuda(e, "colvar_prep");
    } else {
        PrepArgs pa;
        pa.mu_all = mu_all; pa.ldmu = ldmu;
        pa.parts = peers.on() ? peers.mu_parts : nullptr; pa.ld_part = peers.ld_part; pa.rows_per_part = b_loc;
        pa.z = z; pa.ldz = ldz;
        pa.eps = fz.eps; pa.ldeps = fz.ldeps; pa.z_out = fz.z_out; pa.ldz_out = fz.ldz_out;
        pa.mu_loc = peers.on() ? mu_all : mu_all + (int64_t)row_offset * ldmu; pa.ldmu_loc = ldmu;
        pa.logvar = logvar; pa.ldlv = ldlv;
        pa.b_loc = b_loc; pa.b_glob = b_glob; pa.d = d; pa.bl_pad = p.bl_pad; pa.bg_pad = p.bg_pad; pa.dp = p.dp;
        pa.mu_pad = mu_pad; pa.zs = zs; pa.ns = ns; pa.qmax = qmax; pa.shift = shift; pa.vr = vr; pa.ticket = ticket;
        pa.sync = peers.sync;
        if ((e = launch_prep(pa, st)) != cudaSuccess) return fail_cuda(e, "prep");
    }

    FwdArgs fa;
    fa.zs = zs; fa.ns = ns; fa.qmax = qmax; fa.mu_pad = mu_pad;
    fa.s2 = p.save ? at<float>(workspace, p.off_s2) : nullptr; fa.ld_s2 = p.ld_s2;
    fa.Spart = Spart; fa.Jpart = Jpart;
    fa.b_loc = b_loc; fa.bl_pad = p.bl_pad; fa.bg_pad = p.bg_pad; fa.row_offset = row_offset; fa.js_len = p.js_len_fwd;
    fa.seg = p.seg_fwd; fa.n_rb = p.n_rb_fwd;
    fa.w = w;
    int n_js_used = p.n_js_fwd;
    if (p.var_col) {
        if ((e = launch_fwd_colvar(p, fa, &n_js_used, st)) != cudaSuccess) return fail_cuda(e, "tc_fwd_colvar");
    } else {
        if ((e = launch_fwd(p, fa, st)) != cudaSuccess) return fail_cuda(e, "tc_fwd");
    }

    FinArgs fin;
    fin.Spart = Spart; fin.Jpart = Jpart; fin.shift = shift;
    fin.S = at<float>(workspace, p.off_S); fin.J2 = at<float>(workspace, p.off_J2);
    fin.log_qz = log_qz; fin.log_qz_prod = log_qz_prod;
    fin.b_loc = b_loc; fin.bl_pad = p.bl_pad; fin.d = d; fin.dp = p.dp; fin.n_js = n_js_used; fin.lw_u = w.lw_u;
    fin.seg = p.seg_fwd; if (p.var_col) fin.seg.n_ctas = 0;
    fin.tiles_per_block = p.tiles_fwd; fin.rows_per_block = p.fwd_rows;
    fin.lv = nullptr; fin.ldlv = 0; fin.mu_loc = nullptr; fin.ldmu = 0; fin.beta = lf.beta; fin.loss_rows = nullptr; fin.kl_rows = nullptr;
    fin.loss_mean = nullptr; fin.kl_mean = nullptr; fin.rec_rows = nullptr; fin.scale = 0.0f; fin.expelbo = nullptr; fin.e_rows = nullptr;
    fin.red_part = nullptr; fin.ticket = nullptr;
    if (lf.on) {
        fin.lv = logvar; fin.ldlv = ldlv; fin.mu_loc = peers.on() ? mu_all : mu_all + (int64_t)row_offset * ldmu; fin.ldmu = ldmu;
        fin.loss_rows = lf.loss_rows; fin.kl_rows = lf.kl_rows;
        if (fz.loss_mean || fz.kl_mean || fz.expelbo) {
            fin.loss_mean = fz.loss_mean; fin.kl_mean = fz.kl_mean;
            fin.red_part = at<float>(workspace, p.off_red); fin.ticket = ticket;
        }
        if (fz.expelbo) { fin.rec_rows = fz.rec_rows; fin.scale = fz.scale; fin.expelbo = fz.expelbo; fin.e_rows = fz.e_rows; }
    }
    if ((e = launch_fwd_finalize(p, fin, st)) != cudaSuccess) return fail_cuda(e, "fwd_finalize");
    return TCELBO_OK;
}

static int backward_impl(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                         int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                         const float* g_log_qz, const float* g_log_qz_prod, const LossFusion& lf,
                         float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                         const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream,
                         const Peers& peers = Peers()) {
    if (int rc = check_common(z, mu_all, logvar, b_loc, b_glob, row_offset, d, dataset_size, flags, ldz, ldmu, ldlv, true)) return rc;
    if (peers.on() && (flags & TCELBO_VAR_COL)) return fail(TCELBO_ERR_UNSUPPORTED, "the peer-memory exchange covers the row-variance density");
    if (lf.fz.eps && lf.fz.ldeps < d) return fail(TCELBO_ERR_INVALID, "eps row pitch smaller than d");
    if (lf.fz.g_expelbo && !lf.fz.e_rows) return fail(TCELBO_ERR_INVALID, "g_expelbo needs the e_rows the forward wrote");
    if (!(flags & TCELBO_SAVE_FOR_BACKWARD)) return fail(TCELBO_ERR_INVALID, "backward needs the workspace of a forward run with TCELBO_SAVE_FOR_BACKWARD");
    if (!grad_z || !grad_mu_all || !grad_logvar) return fail(TCELBO_ERR_INVALID, "null gradient pointer");
    if (!lf.on && (!g_log_qz || !g_log_qz_prod)) return fail(TCELBO_ERR_INVALID, "null upstream gradient pointer");
    if (ldgz < d || ldgmu < d || ldglv < d) return fail(TCELBO_ERR_INVALID, "gradient row pitch smaller than d");
    Plan p;
    if (!make_plan(p, b_loc, b_glob, d, flags, sm_count())) return fail(TCELBO_ERR_INVALID, "cannot plan this shape");
    if (!workspace || workspace_bytes < p.total_bytes || !aligned256(workspace))
        return fail(TCELBO_ERR_WORKSPACE, "workspace must be the %zu-byte buffer forward wrote (got %zu)", p.total_bytes, workspace_bytes);
    if (!scratch || scratch_bytes < p.bwd_bytes || !aligned256(scratch))
        return fail(TCELBO_ERR_WORKSPACE, "scratch must be 256-byte aligned and at least %zu bytes (got %zu)", p.bwd_bytes, scratch_bytes);
    if (lf.on && p.var_col) return fail(TCELBO_ERR_INVALID, "the fused loss uses the row-variance density");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Weights w = make_weights(b_glob, dataset_size, flags);
    cudaError_t e;

    void* wsm = const_cast<void*>(workspace);                       // only read below
    const float* mu_pad = at<float>(wsm, p.off_mu);
    const float* zs = at<float>(wsm, p.off_zs);
    const float* ns = at<float>(wsm, p.off_ns);
    const float* qmax = at<float>(wsm, p.off_qmax);
    const float* vr = at<float>(wsm, p.off_vr);
    const float* S = at<float>(wsm, p.off_S);
    const float* J2 = at<float>(wsm, p.off_J2);
    const float* s2 = at<float>(wsm, p.off_s2);
    float* gps = at<float>(scratch, p.boff_gps);
    float* gj = at<float>(scratch, p.boff_gj);
    float* gk = at<float>(scratch, p.boff_gk);
    float* Apart = at<float>(scratch, p.boff_A);
    float* CRpart = at<float>(scratch, p.boff_CR);
    float* Gpart = at<float>(scratch, p.boff_G);

    const size_t zero_n = (size_t)(p.var_col ? 2 : 1) * p.bg_pad * p.dp;
    BwdUpstream up;
    up.g_log_qz = g_log_qz; up.g_log_qz_prod = g_log_qz_prod; up.g_loss = lf.g_loss; up.g_kl = lf.g_kl;
    up.g_loss_mean = lf.fz.g_loss_mean; up.g_kl_mean = lf.fz.g_kl_mean; up.g_expelbo = lf.fz.g_expelbo; up.e_rows = lf.fz.e_rows;
    up.scale = lf.fz.scale; up.g_rec_rows = lf.fz.g_rec_rows; up.beta = lf.beta;
    up.epoch = (peers.on() && peers.sync.on()) ? peers.sync.state + 1 : nullptr;
    if ((peers.phase & 1) && (e = launch_bwd_prep(p, up, S, gps, gj, lf.on ? gk : nullptr, Gpart, zero_n, st)) != cudaSuccess)
        return fail_cuda(e, "bwd_prep");

    BwdFinArgs fa;
    fa.Apart = Apart; fa.CRpart = CRpart; fa.Gpart = Gpart; fa.ns = ns; fa.vr = vr;
    fa.grad_z = grad_z; fa.ldgz = ldgz; fa.grad_lv = grad_logvar; fa.ldglv = ldglv; fa.grad_mu = grad_mu_all; fa.ldgmu = ldgmu;
    fa.b_loc = b_loc; fa.b_glob = b_glob; fa.bl_pad = p.bl_pad; fa.bg_pad = p.bg_pad; fa.d = d; fa.dp = p.dp;
    fa.n_js = 1; fa.n_is = 1;
    fa.seg = Segments{0, 0, 0}; fa.tiles_per_block = 0; fa.n_rb = 0; fa.rows_per_block = 0; fa.slice_dp = 0;
    fa.gk = lf.on ? gk : nullptr; fa.lv = logvar; fa.ldlv = ldlv; fa.mu_all = mu_all; fa.ldmu = ldmu; fa.row_offset = row_offset;
    fa.scratch_parts = peers.on() ? peers.scratch_parts : nullptr; fa.g_off = p.boff_G; fa.n_ranks = peers.n_ranks;
    fa.eps = lf.fz.eps; fa.ldeps = lf.fz.ldeps;
    fa.sync = peers.sync;

    BwdFusedArgs ua;
    ua.zs = zs; ua.ns = ns; ua.qmax = qmax; ua.gps = gps; ua.gj = gj; ua.J2 = J2; ua.mu_pad = mu_pad;
    ua.s2 = s2; ua.ld_s2 = p.ld_s2; ua.Apart = Apart; ua.CRpart = CRpart; ua.Gacc = Gpart; ua.Gacc2 = nullptr;
    ua.b_loc = b_loc; ua.bl_pad = p.bl_pad; ua.bg_pad = p.bg_pad; ua.row_offset = row_offset; ua.js_len = 0; ua.w = w;
    ua.seg = Segments{0, 0, 0}; ua.n_blocks = 0; ua.n_rb = 0;
    ua.plan_only = (peers.phase & 1) ? 0 : 1;

    if (p.var_col) {
        float* Glv = Gpart + (size_t)p.bg_pad * p.dp;
        ua.Gacc2 = Glv;
        if ((e = launch_bwd_colvar(p, ua, &fa.n_js, st)) != cudaSuccess) return fail_cuda(e, "tc_bwd_colvar");
        if ((e = launch_bwd_colvar_finalize(p, fa, mu_pad, Glv, st)) != cudaSuccess) return fail_cuda(e, "bwd_colvar_finalize");
        return TCELBO_OK;
    }
    // single fused sweep: row-local sums in registers, column sums via smem staging + red.global
    if ((e = launch_bwd_fused(p, ua, &fa, st)) != cudaSuccess) return fail_cuda(e, "tc_bwd_fused");
    if (!(peers.phase & 2)) return TCELBO_OK;
    if ((e = launch_bwd_fused_finalize(p, fa, st)) != cudaSuccess) return fail_cuda(e, "bwd_fused_finalize");
    return TCELBO_OK;
}

int tcelbo_forward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                   int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                   float* log_qz, float* log_qz_prod, void* workspace, size_t workspace_bytes, void* stream) {
    return forward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                        log_qz, log_qz_prod, LossFusion(), workspace, workspace_bytes, stream);
}

int tcelbo_backward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                    int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags,
                    const float* g_log_qz, const float* g_log_qz_prod,
                    float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                    const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream) {
    return backward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                         g_log_qz, g_log_qz_prod, LossFusion(), grad_z, ldgz, grad_mu_all, ldgmu, grad_logvar, ldglv,
                         workspace, workspace_bytes, scratch, scratch_bytes, stream);
}

int tcelbo_klloss_forward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                          int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                          float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod,
                          void* workspace, size_t workspace_bytes, void* stream) {
    if (!loss_rows || !kl_rows) return fail(TCELBO_ERR_INVALID, "null output pointer");
    LossFusion lf; lf.on = true; lf.beta = beta; lf.loss_rows = loss_rows; lf.kl_rows = kl_rows;
    return forward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                        log_qz, log_qz_prod, lf, workspace, workspace_bytes, stream);
}

int tcelbo_klloss_backward(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                           int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                           const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                           float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                           const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream) {
    if (!g_loss_rows) return fail(TCELBO_ERR_INVALID, "null upstream gradient pointer");
    LossFusion lf; lf.on = true; lf.beta = beta; lf.g_loss = g_loss_rows; lf.g_kl = g_kl_rows;
    return backward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                         g_log_qz, g_log_qz_prod, lf, grad_z, ldgz, grad_mu_all, ldgmu, grad_logvar, ldglv,
                         workspace, workspace_bytes, scratch, scratch_bytes, stream);
}

int tcelbo_klloss_forward_ex(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                             int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                             float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod, const tcelbo_fusion* fusion,
                             void* workspace, size_t workspace_bytes, void* stream) {
    if (!loss_rows || !kl_rows) return fail(TCELBO_ERR_INVALID, "null output pointer");
    LossFusion lf; lf.on = true; lf.beta = beta; lf.loss_rows = loss_rows; lf.kl_rows = kl_rows;
    if (fusion) lf.fz = *fusion;
    return forward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                        log_qz, log_qz_prod, lf, workspace, workspace_bytes, stream);
}

int tcelbo_klloss_backward_ex(const float* z, int64_t ldz, const float* mu_all, int64_t ldmu, const float* logvar, int64_t ldlv,
                              int b_loc, int b_glob, int row_offset, int d, int64_t dataset_size, uint32_t flags, float beta,
                              const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                              const tcelbo_fusion* fusion,
                              float* grad_z, int64_t ldgz, float* grad_mu_all, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                              const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes, void* stream) {
    LossFusion lf; lf.on = true; lf.beta = beta; lf.g_loss = g_loss_rows; lf.g_kl = g_kl_rows;
    if (fusion) lf.fz = *fusion;
    if (!g_loss_rows && !lf.fz.g_loss_mean && !lf.fz.g_expelbo && !g_kl_rows && !lf.fz.g_kl_mean && !g_log_qz && !g_log_qz_prod)
        return fail(TCELBO_ERR_INVALID, "no upstream gradient given");
    return backward_impl(z, ldz, mu_all, ldmu, logvar, ldlv, b_loc, b_glob, row_offset, d, dataset_size, flags,
                         g_log_qz, g_log_qz_prod, lf, grad_z, ldgz, grad_mu_all, ldgmu, grad_logvar, ldglv,
                         workspace, workspace_bytes, scratch, scratch_bytes, stream);
}

int tcelbo_klloss_forward_peer(const float* z, int64_t ldz, const float* mu_loc, int64_t ldmu, const float* const* mu_parts, int64_t ld_part,
                               const float* logvar, int64_t ldlv, int b_loc, int n_ranks, int rank, int d, int64_t dataset_size,
                               uint32_t flags, float beta, float* loss_rows, float* kl_rows, float* log_qz, float* log_qz_prod,
                               const tcelbo_fusion* fusion, const tcelbo_peer_sync* sync, void* workspace, size_t workspace_bytes, void* stream) {
    if (!loss_rows || !kl_rows || !mu_parts) return fail(TCELBO_ERR_INVALID, "null pointer");
    if (sync && (!sync->flag_parts || !sync->state)) return fail(TCELBO_ERR_INVALID, "peer_sync needs the flag table and the state words");
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks || ld_part < d) return fail(TCELBO_ERR_INVALID, "bad rank / n_ranks / ld_part");
    if ((int64_t)b_loc * n_ranks > INT32_MAX) return fail(TCELBO_ERR_INVALID, "global batch too large");
    LossFusion lf; lf.on = true; lf.beta = beta; lf.loss_rows = loss_rows; lf.kl_rows = kl_rows;
    if (fusion) lf.fz = *fusion;
    Peers peers; peers.mu_parts = mu_parts; peers.ld_part = ld_part; peers.n_ranks = n_ranks;
    if (sync) peers.sync = PeerSync{sync->flag_parts, sync->state, 0, rank, n_ranks};
    return forward_impl(z, ldz, mu_loc, ldmu, logvar, ldlv, b_loc, b_loc * n_ranks, rank * b_loc, d, dataset_size, flags,
                        log_qz, log_qz_prod, lf, workspace, workspace_bytes, stream, peers);
}

int tcelbo_peer_publish(const float* mu_loc, int64_t ldmu, int b_loc, int d, float* published, const tcelbo_peer_sync* sync, void* stream) {
    if (!mu_loc || !published || b_loc < 1 || d < 1 || ldmu < d) return fail(TCELBO_ERR_INVALID, "bad argument");
    if (sync && !sync->state) return fail(TCELBO_ERR_INVALID, "peer_sync needs the state words");
    cudaError_t e = launch_publish(mu_loc, ldmu, b_loc, d, published, sync ? sync->state : nullptr, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "publish");
}

int tcelbo_klloss_backward_peer(int phase, const float* z, int64_t ldz, const float* mu_loc, int64_t ldmu, const float* logvar, int64_t ldlv,
                                int b_loc, int n_ranks, int rank, int d, int64_t dataset_size, uint32_t flags, float beta,
                                const float* g_loss_rows, const float* g_kl_rows, const float* g_log_qz, const float* g_log_qz_prod,
                                float* grad_z, int64_t ldgz, float* grad_mu_loc, int64_t ldgmu, float* grad_logvar, int64_t ldglv,
                                const void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                                const void* const* scratch_parts, const tcelbo_fusion* fusion, const tcelbo_peer_sync* sync, void* stream) {
    if (sync && (!sync->flag_parts || !sync->state)) return fail(TCELBO_ERR_INVALID, "peer_sync needs the flag table and the state words");
    if (!g_loss_rows && !(fusion && (fusion->g_loss_mean || fusion->g_expelbo || fusion->g_kl_mean)) && !g_kl_rows && !g_log_qz && !g_log_qz_prod)
        return fail(TCELBO_ERR_INVALID, "no upstream gradient given");
    if (phase != TCELBO_PEER_SWEEP && phase != TCELBO_PEER_FINISH) return fail(TCELBO_ERR_INVALID, "phase must be TCELBO_PEER_SWEEP or TCELBO_PEER_FINISH");
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(TCELBO_ERR_INVALID, "bad rank / n_ranks");
    if (phase == TCELBO_PEER_FINISH && !scratch_parts) return fail(TCELBO_ERR_INVALID, "null scratch table");
    if ((int64_t)b_loc * n_ranks > INT32_MAX) return fail(TCELBO_ERR_INVALID, "global batch too large");
    LossFusion lf; lf.on = true; lf.beta = beta; lf.g_loss = g_loss_rows; lf.g_kl = g_kl_rows;
    if (fusion) lf.fz = *fusion;
    Peers peers; peers.scratch_parts = scratch_parts; peers.n_ranks = n_ranks; peers.phase = phase;
    if (sync) peers.sync = PeerSync{sync->flag_parts, sync->state, 1, rank, n_ranks};
    return backward_impl(z, ldz, mu_loc, ldmu, logvar, ldlv, b_loc, b_loc * n_ranks, rank * b_loc, d, dataset_size, flags,
                         g_log_qz, g_log_qz_prod, lf, grad_z, ldgz, grad_mu_loc, ldgmu, grad_logvar, ldglv,
                         workspace, workspace_bytes, scratch, scratch_bytes, stream, peers);
}

#define ROWOP_CHECK(cond, msg) do { if (!(cond)) return fail(TCELBO_ERR_INVALID, msg); } while (0)

int tcelbo_kl_forward(const float* logvar, int64_t ldlv, const float* mu, int64_t ldmu, int b, int d, float* kl_rows, void* stream) {
    ROWOP_CHECK(logvar && mu && kl_rows, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldlv >= d && ldmu >= d, "bad shape");
    cudaError_t e = launch_kl_fwd(logvar, ldlv, mu, ldmu, b, d, kl_rows, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "kl_fwd");
}

int tcelbo_kl_backward(const float* logvar, int64_t ldlv, const float* mu, int64_t ldmu, const float* g_rows, int b, int d,
                       float* grad_logvar, int64_t ldglv, float* grad_mu, int64_t ldgmu, void* stream) {
    ROWOP_CHECK(logvar && mu && g_rows && grad_logvar && grad_mu, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldlv >= d && ldmu >= d && ldglv >= d && ldgmu >= d, "bad shape");
    cudaError_t e = launch_kl_bwd(logvar, ldlv, mu, ldmu, g_rows, b, d, grad_logvar, ldglv, grad_mu, ldgmu, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "kl_bwd");
}

int tcelbo_reparam_forward(const float* mu, int64_t ldmu, const float* logvar, int64_t ldlv, const float* eps, int64_t ldeps,
                           int b, int d, float* z, int64_t ldz, void* stream) {
    ROWOP_CHECK(mu && logvar && eps && z, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldmu >= d && ldlv >= d && ldeps >= d && ldz >= d, "bad shape");
    cudaError_t e = launch_reparam_fwd(mu, ldmu, logvar, ldlv, eps, ldeps, b, d, z, ldz, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "reparam_fwd");
}

int tcelbo_reparam_backward(const float* logvar, int64_t ldlv, const float* eps, int64_t ldeps, const float* g_z, int64_t ldgz,
                            int b, int d, float* grad_mu, int64_t ldgmu, float* grad_logvar, int64_t ldglv, void* stream) {
    ROWOP_CHECK(logvar && eps && g_z && grad_mu && grad_logvar, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldlv >= d && ldeps >= d && ldgz >= d && ldgmu >= d && ldglv >= d, "bad shape");
    cudaError_t e = launch_reparam_bwd(logvar, ldlv, eps, ldeps, g_z, ldgz, b, d, grad_mu, ldgmu, grad_logvar, ldglv, false, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "reparam_bwd");
}

int tcelbo_reparam_backward_acc(const float* logvar, int64_t ldlv, const float* eps, int64_t ldeps, const float* g_z, int64_t ldgz,
                            int b, int d, float* grad_mu, int64_t ldgmu, float* grad_logvar, int64_t ldglv, void* stream) {
    ROWOP_CHECK(logvar && eps && g_z && grad_mu && grad_logvar, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldlv >= d && ldeps >= d && ldgz >= d && ldgmu >= d && ldglv >= d, "bad shape");
    cudaError_t e = launch_reparam_bwd(logvar, ldlv, eps, ldeps, g_z, ldgz, b, d, grad_mu, ldgmu, grad_logvar, ldglv, true, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "reparam_bwd");
}

int tcelbo_rowdensity_forward(const float* x, int64_t ldx, const float* mu, int64_t ldmu, const float* logvar, int64_t ldlv,
                              int b, int d, float* out, void* stream) {
    ROWOP_CHECK(x && out, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldx >= d && (!mu || ldmu >= d) && (!logvar || ldlv >= d), "bad shape");
    cudaError_t e = launch_rowdensity_fwd(x, ldx, mu, ldmu, logvar, ldlv, b, d, out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "rowdensity_fwd");
}

int tcelbo_rowdensity_backward(const float* x, int64_t ldx, const float* mu, int64_t ldmu, const float* logvar, int64_t ldlv,
                               const float* g_rows, int b, int d, float* grad_x, int64_t ldgx, float* grad_mu, int64_t ldgmu,
                               float* grad_logvar, int64_t ldglv, void* stream) {
    ROWOP_CHECK(x && g_rows, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && ldx >= d && (!mu || ldmu >= d) && (!logvar || ldlv >= d), "bad shape");
    ROWOP_CHECK((!grad_x || ldgx >= d) && (!grad_mu || ldgmu >= d) && (!grad_logvar || ldglv >= d), "bad gradient pitch");
    cudaError_t e = launch_rowdensity_bwd(x, ldx, mu, ldmu, logvar, ldlv, g_rows, b, d, grad_x, ldgx, grad_mu, ldgmu,
                                          grad_logvar, ldglv, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "rowdensity_bwd");
}

int tcelbo_recloss_chunks(int b, int64_t n) {
    int c = (int)((n + 4095) / 4096);                       // ~4K pixels per CTA, enough CTAs to fill the GPU at small batches
    const int want = (148 * 4 + b - 1) / (b > 0 ? b : 1);
    if (c > want) c = want;
    if (c < 1) c = 1;
    return c;
}

int tcelbo_recloss_forward(const float* x, const float* recon, int b, int64_t n, int kind, float* partial, float* out_rows, void* stream) {
    ROWOP_CHECK(x && recon && partial && out_rows, "null pointer");
    ROWOP_CHECK(b >= 1 && n >= 1 && kind >= 0 && kind <= 2, "bad argument");
    cudaError_t e = launch_recloss_fwd(x, recon, b, n, kind, partial, tcelbo_recloss_chunks(b, n), out_rows, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "recloss_fwd");
}

int tcelbo_recloss_backward(const float* x, const float* recon, const float* g_rows, int b, int64_t n, int kind, float* grad_recon, void* stream) {
    ROWOP_CHECK(x && recon && g_rows && grad_recon, "null pointer");
    ROWOP_CHECK(b >= 1 && n >= 1 && kind >= 0 && kind <= 2, "bad argument");
    cudaError_t e = launch_recloss_bwd(x, recon, g_rows, b, n, kind, grad_recon, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "recloss_bwd");
}

int tcelbo_expelbo_forward(const float* rec_rows, const float* kl_rows, int b, float scale, float* out, float* e_rows, void* stream) {
    ROWOP_CHECK(rec_rows && kl_rows && out && e_rows && b >= 1, "bad argument");
    cudaError_t e = launch_expelbo_fwd(rec_rows, kl_rows, b, scale, out, e_rows, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "expelbo_fwd");
}

int tcelbo_expelbo_backward(const float* e_rows, const float* g_out, int b, float scale, float* g_rows, void* stream) {
    ROWOP_CHECK(e_rows && g_out && g_rows && b >= 1, "bad argument");
    cudaError_t e = launch_expelbo_bwd(e_rows, g_out, b, scale, g_rows, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "expelbo_bwd");
}

int tcelbo_density_forward(int floored, const float* x, const float* mu, const float* logvar, const int64_t* shape,
                           const int64_t* sx, const int64_t* sm, const int64_t* sl, float* out, void* stream) {
    ROWOP_CHECK(x && mu && logvar && out && shape && sx && sm && sl, "null pointer");
    ROWOP_CHECK(shape[0] >= 1 && shape[1] >= 1 && shape[2] >= 1, "bad shape");
    cudaError_t e = launch_density_fwd(floored != 0, x, mu, logvar, shape, sx, sm, sl, out, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "density_fwd");
}

int tcelbo_density_backward(int floored, const float* x, const float* mu, const float* logvar, const float* g, const int64_t* shape,
                            const int64_t* sx, const int64_t* sm, const int64_t* sl, float* gx, float* gmu, float* glv, void* stream) {
    ROWOP_CHECK(x && mu && logvar && g && gx && gmu && glv && shape && sx && sm && sl, "null pointer");
    cudaError_t e = launch_density_bwd(floored != 0, x, mu, logvar, g, shape, sx, sm, sl, gx, gmu, glv, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "density_bwd");
}

namespace {
void sampling_weights(int b, int64_t n, uint32_t flags, Weights& w, float& lw_n, float& lw_s, float& post) {
    w = make_weights(b, n, flags);
    lw_n = lw_s = 0.0f; post = 0.0f;
    if (flags & TCELBO_EST_MWS) { post = w.lw_u; return; }                    // subtract log(B*N) after the logsumexp
    const double m = (double)(b - 1);
    lw_n = logf((float)(1.0 / (double)n));
    lw_s = logf((float)(((double)n - m) / ((double)n * m)));                  // NaN when N < B-1, like the reference
}
}  // namespace

int tcelbo_sampling_forward(const float* log_qz_prob, int b, int d, int64_t dataset_size, uint32_t flags,
                            float* log_qz_prod, float* log_qz, float* lse_dim, float* pair_sums, void* stream) {
    ROWOP_CHECK(log_qz_prob && log_qz_prod && log_qz && lse_dim && pair_sums, "null pointer");
    ROWOP_CHECK(b >= 1 && d >= 1 && dataset_size >= 1, "bad shape");
    if (b < 2 && !(flags & TCELBO_EST_MWS)) return fail(TCELBO_ERR_INVALID, "b == 1: the stratified weight divides by B-1 (ops.py:44)");
    Weights w; float lw_n, lw_s, post;
    sampling_weights(b, dataset_size, flags, w, lw_n, lw_s, post);
    cudaError_t e = launch_sampling_fwd(log_qz_prob, b, d, w, lw_n, lw_s, post, log_qz_prod, log_qz, lse_dim, pair_sums, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "sampling_fwd");
}

int tcelbo_sampling_backward(const float* log_qz_prob, int b, int d, int64_t dataset_size, uint32_t flags,
                             const float* g_log_qz_prod, const float* g_log_qz, const float* lse_dim, const float* pair_sums,
                             const float* log_qz, float* grad_log_qz_prob, void* stream) {
    ROWOP_CHECK(log_qz_prob && g_log_qz_prod && g_log_qz && lse_dim && pair_sums && log_qz && grad_log_qz_prob, "null pointer");
    Weights w; float lw_n, lw_s, post;
    sampling_weights(b, dataset_size, flags, w, lw_n, lw_s, post);
    cudaError_t e = launch_sampling_bwd(log_qz_prob, b, d, w, lw_n, lw_s, post, g_log_qz_prod, g_log_qz, lse_dim, pair_sums, log_qz,
                                        grad_log_qz_prob, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "sampling_bwd");
}

long long tcelbo_launch_count(void) { return instr().launches.load(); }

int tcelbo_profile_events(int kernel_id, void* start_event, void* stop_event) {
    if (kernel_id < 0 || kernel_id > 3) return fail(TCELBO_ERR_INVALID, "kernel_id must be 0..3");
    Instr& in = instr();
    in.timed_kernel = kernel_id;
    in.ev_start = static_cast<cudaEvent_t>(start_event);
    in.ev_stop = static_cast<cudaEvent_t>(stop_event);
    return TCELBO_OK;
}

int tcelbo_ex2_peak(float* scratch, int iters, int ctas, void* stream) {
    ROWOP_CHECK(scratch && iters > 0 && ctas > 0, "bad argument");
    cudaError_t e = launch_ex2_peak(scratch, iters, ctas, static_cast<cudaStream_t>(stream));
    return e == cudaSuccess ? TCELBO_OK : fail_cuda(e, "ex2_peak");
}

}  // extern "C"
