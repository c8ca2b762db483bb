// Column-variance variant of the TC estimator: log q(z_i | mu_j, var_j) with the un-floored density of
// ops.py:24-29 as it is called at solvers/tc.py:114-116 (the reference's "full" MI/TC/dim-KL path).
//
//   per (j,d)   sj = sqrt(0.5*log2e*exp(-lv_j)), nmus = -mu_j*sj, c2 = -0.5*(lv_j + log 2pi)*log2e
//   per (i,j,d) dl = z_i*sj + nmus ; t = c2 - dl^2 ; tcl = max(t, -50*log2e) ; e = 2^tcl     (lp = ln2 * tcl)
//   S_id = sum_j rho_ij e ; s2_ij = -sum_d tcl ; J2_i = log2 sum_j rho_ij 2^(-s2_ij)
//   backward  r = (gJ_i q_ij + gP_i rho e / S_id) [t >= -50 log2e]
//             grad_z[i,d]  = -2 ln2 sum_j r dl sj        (row-local)
//             grad_mu[j,d] =  2 ln2 sj sum_i r dl         (column sum)
//             grad_lv[j,d] =  sum_i r (ln2 dl^2 - 0.5)    (column sum)
// Same machinery as the row-variance kernels (bulk-TMA column pipeline, rows in registers, column sums
// staged through shared memory), but three column operands are streamed instead of one.  This is the
// reference's dead-code path, so it is built for correctness first and shares the tuned kernels' layout.
#include "tc_common.cuh"
#include "tc_kernels.h"
#include "tc_instr.h"

namespace tcelbo {

__device__ __forceinline__ void red_add_v4_cv(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// (sj, nmus, c2) of one column element, shared by the plain and the peer-gather prologue so that both pack the same bits
__device__ __forceinline__ void colpack_of(float m, float lv, float& sj, float& nmus, float& c2) {
    const float iv = expf(-lv);
    sj = sqrtf(0.5f * kLog2e * iv);
    c2 = -0.5f * (lv + kLog2Pi) * kLog2e;
    // logvar < -88.7: exp(-logvar) is +inf in fp32, so ops.py:27-29 yields -inf -> -50 for every z != mu.  Keep that
    // behaviour with finite operands (dl^2 overflows to +inf and the clamp takes over) instead of inf - inf = NaN,
    // and keep the unshifted sum S = sum_j rho 2^t finite: c2 stays <= 63 for every column that can be unclamped.
    if (isinf(iv)) { sj = 1.0e19f; c2 = 0.0f; }
    nmus = -(m * sj);
}

// column operands: colpack[j][0..2][dp] = (sj, nmus, c2); rows: zpad[i][dp] (zero padded), shift[i][dp] = 0; zeroes the
// ticket of the finalize kernel's batch means (the workspace may be fresh, uninitialised memory).  kParts: the columns live in
// b_loc-row blocks of different allocations (one per rank, peer-mapped); the rows (local data) are written first, then the
// in-kernel barrier waits for every rank's publish, then the columns are gathered with volatile loads, V (1 or 4) dims per thread.
// With eps the local rows of z are formed here from mu_loc / lv_loc (fused reparameterize) and stored to z_out if given.
template <bool kParts, int V>
__global__ void colvar_prep_kernel(const ColPrepArgs a) {
    const int64_t n_row = (int64_t)a.bl_pad * a.dp;
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.ticket = 0u;
    for (int64_t k = t0; k < n_row; k += stride) {
        const int i = (int)(k / a.dp), dd = (int)(k % a.dp);
        float zv = 0.0f;
        if (i < a.b_loc && dd < a.d) {
            if (a.eps != nullptr) {
                zv = reparam_z(a.mu_loc[(int64_t)i * a.ldmu + dd], a.lv_loc[(int64_t)i * a.ldlv + dd], a.eps[(int64_t)i * a.ldeps + dd]);
                if (a.z_out != nullptr) a.z_out[(int64_t)i * a.ldz_out + dd] = zv;
            } else {
                zv = a.z[(int64_t)i * a.ldz + dd];
            }
        }
        a.zpad[k] = zv;
        a.shift[k] = 0.0f;
    }
    if (kParts && a.sync.on()) peer_barrier(a.sync);
    const int dpv = a.dp / V;
    const int64_t n_col = (int64_t)a.bg_pad * dpv;
    for (int64_t idx = t0; idx < n_col; idx += stride) {
        const int j = (int)(idx / dpv), dd = V * (int)(idx % dpv);
        float m[V], l[V];
        if (kParts && j < a.b_glob && dd < a.d) {
            const int part = j / a.b_loc;
            const int64_t o = (int64_t)(j - part * a.b_loc) * a.ld_part + dd;
            if (V == 4) {                                        // d % 4 == 0: dd < d covers all four
                const float4 mv = ld_volatile_v4(a.mu_parts[part] + o), lv = ld_volatile_v4(a.lv_parts[part] + o);
                m[0] = mv.x; m[1] = mv.y; m[2] = mv.z; m[3] = mv.w;
                l[0] = lv.x; l[1] = lv.y; l[2] = lv.z; l[3] = lv.w;
            } else {
                m[0] = *static_cast<const volatile float*>(a.mu_parts[part] + o);
                l[0] = *static_cast<const volatile float*>(a.lv_parts[part] + o);
            }
        } else if (!kParts && j < a.b_glob && dd < a.d) {
#pragma unroll
            for (int e = 0; e < V; ++e) { m[e] = a.mu_all[(int64_t)j * a.ldmu + dd + e]; l[e] = a.lv_all[(int64_t)j * a.ldlv + dd + e]; }
        }
        float sj[V], nmus[V], c2[V];
#pragma unroll
        for (int e = 0; e < V; ++e) {
            sj[e] = 0.f; nmus[e] = 0.f; c2[e] = 0.f;
            if (j < a.b_glob && dd + e < a.d) colpack_of(m[e], l[e], sj[e], nmus[e], c2[e]);
        }
        float* o = a.colpack + (size_t)j * 3 * a.dp + dd;
        if (V == 4) {
            *reinterpret_cast<float4*>(o) = make_float4(sj[0], sj[1], sj[2], sj[3]);
            *reinterpret_cast<float4*>(o + a.dp) = make_float4(nmus[0], nmus[1], nmus[2], nmus[3]);
            *reinterpret_cast<float4*>(o + 2 * a.dp) = make_float4(c2[0], c2[1], c2[2], c2[3]);
        } else {
            o[0] = sj[0]; o[a.dp] = nmus[0]; o[2 * a.dp] = c2[0];
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// forward: LPR lanes share a row, 32 dims per lane (same mapping as tc_fwd_kernel)
// ------------------------------------------------------------------------------------------------------
template <int LPR> struct CvGeom {
    static constexpr int DP = 32 * LPR;
    static constexpr int JT0 = (kTileFloats / DP) > 32 ? 32 : (kTileFloats / DP);
    static constexpr int JT = (JT0 / 4) < 4 ? 4 : (JT0 / 4);            // columns per stage (three operands each)
    static constexpr int TILE = JT * 3 * DP;
};

template <int LPR, bool kWeighted>
__device__ __forceinline__ float cv_fwd_one_column(const float* __restrict__ col, const u64 (&z2)[16], u64 (&S2)[16], float rho) {
    constexpr int DP = 32 * LPR;
    u64 acc0 = 0ull, acc1 = 0ull;
    const u64 rho2 = pack2(rho, rho);
    const u64 neg1 = pack2(-1.0f, -1.0f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float4 s = *reinterpret_cast<const float4*>(col + 4 * LPR * k);
        const float4 n = *reinterpret_cast<const float4*>(col + DP + 4 * LPR * k);
        const float4 c = *reinterpret_cast<const float4*>(col + 2 * DP + 4 * LPR * k);
        const u64 d01 = ffma2(z2[2 * k], pack2(s.x, s.y), pack2(n.x, n.y));
        const u64 d23 = ffma2(z2[2 * k + 1], pack2(s.z, s.w), pack2(n.z, n.w));
        const u64 t01 = ffma2(fmul2(d01, d01), neg1, pack2(c.x, c.y));
        const u64 t23 = ffma2(fmul2(d23, d23), neg1, pack2(c.z, c.w));
        float t0, t1, t2, t3;
        unpack2(t01, t0, t1); unpack2(t23, t2, t3);
        t0 = fmax_nan(t0, -kK50); t1 = fmax_nan(t1, -kK50); t2 = fmax_nan(t2, -kK50); t3 = fmax_nan(t3, -kK50);
        u64 e01 = pack2(ex2(t0), ex2(t1));
        u64 e23 = pack2(ex2(t2), ex2(t3));
        if (kWeighted) { e01 = fmul2(e01, rho2); e23 = fmul2(e23, rho2); }
        S2[2 * k] = fadd2(S2[2 * k], e01);
        S2[2 * k + 1] = fadd2(S2[2 * k + 1], e23);
        acc0 = fadd2(acc0, pack2(t0, t1));
        acc1 = fadd2(acc1, pack2(t2, t3));
    }
    acc0 = fadd2(acc0, acc1);
    float a, b; unpack2(acc0, a, b);
    return -(a + b);                                       // s2 = -sum_d tcl, so that x = log2(rho) - s2 as in the row variant
}

template <int LPR>
__global__ void __launch_bounds__(kFwdWarps * 32, kColvarFwdRes)
tc_fwd_colvar_kernel(const FwdArgs a) {
    using GEO = CvGeom<LPR>;
    constexpr int DP = GEO::DP, JT = GEO::JT, TILE = GEO::TILE;
    constexpr int RPW = 32 / LPR, ROWS = kFwdWarps * RPW;
    constexpr int G = LPR < 4 ? LPR : 4;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tiles = reinterpret_cast<float*>(smem_raw);
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * TILE * sizeof(float));
    uint64_t* bar_empty = bar_full + kStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int l = lane % LPR, rw = lane / LPR;
    const int row = blockIdx.x * ROWS + warp * RPW + rw;
    const int i_glob = a.row_offset + row;

    u64 z2[16], S2[16];
    {
        const float* pz = a.zs + (size_t)row * DP + 4 * l;      // a.zs holds the zero-padded z here
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float4 vz = __ldg(reinterpret_cast<const float4*>(pz + 4 * LPR * k));
            z2[2 * k] = pack2(vz.x, vz.y); z2[2 * k + 1] = pack2(vz.z, vz.w);
            S2[2 * k] = 0ull; S2[2 * k + 1] = 0ull;
        }
    }
    float lse_m = kNegBig, lse_s = 0.0f;
    const int j0 = blockIdx.y * a.js_len;
    const int j1 = min(a.bg_pad, j0 + a.js_len);
    const int ntiles = (j1 - j0) / JT;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], kFwdWarps); }
        mbar_fence_init();
    }
    __syncthreads();
    if (threadIdx.x == 0 && ntiles > 0) {
        mbar_arrive_expect_tx(&bar_full[0], TILE * sizeof(float));
        bulk_g2s(tiles, a.mu_pad + (size_t)j0 * 3 * DP, TILE * sizeof(float), &bar_full[0]);
    }
    float* s2_row = (a.s2 != nullptr) ? a.s2 + (size_t)row * a.ld_s2 : nullptr;

    for (int t = 0; t < ntiles; ++t) {
        const int st = t % kStages;
        if (threadIdx.x == 0 && t + 1 < ntiles) {
            const int sn = (t + 1) % kStages;
            if (t + 1 >= kStages) mbar_wait(&bar_empty[sn], (((t + 1) / kStages) - 1) & 1);
            mbar_arrive_expect_tx(&bar_full[sn], TILE * sizeof(float));
            bulk_g2s(tiles + (size_t)sn * TILE, a.mu_pad + (size_t)(j0 + (t + 1) * JT) * 3 * DP, TILE * sizeof(float), &bar_full[sn]);
        }
        mbar_wait(&bar_full[st], (t / kStages) & 1);
        const float* tile = tiles + (size_t)st * TILE;
        const int jt0 = j0 + t * JT;
        const bool special = (a.w.mss && jt0 == 0) || (jt0 + JT > a.w.b_glob);
        for (int jj = 0; jj < JT; jj += 4) {
            float part[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float rho = 1.0f, l2 = 0.0f;
                if (special) {
                    weight_of(a.w, i_glob, jt0 + jj + u, rho, l2);
                    part[u] = cv_fwd_one_column<LPR, true>(tile + (size_t)(jj + u) * 3 * DP + 4 * l, z2, S2, rho);
                } else {
                    part[u] = cv_fwd_one_column<LPR, false>(tile + (size_t)(jj + u) * 3 * DP + 4 * l, z2, S2, rho);
                }
            }
#pragma unroll
            for (int o = 1; o < LPR; o <<= 1) {
#pragma unroll
                for (int u = 0; u < 4; ++u) part[u] += __shfl_xor_sync(0xffffffffu, part[u], o);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if ((u & (G - 1)) == (l & (G - 1))) {
                    const int j = jt0 + jj + u;
                    float x = -part[u];
                    if (special) { float rho, l2; weight_of(a.w, i_glob, j, rho, l2); x += l2; }
                    lse2_push(lse_m, lse_s, x);
                    if (s2_row != nullptr && l < G) s2_row[j] = part[u];
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_empty[st]);
    }
    {
        float* ps = a.Spart + ((size_t)blockIdx.y * a.bl_pad + row) * DP + 4 * l;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float4 v;
            unpack2(S2[2 * k], v.x, v.y); unpack2(S2[2 * k + 1], v.z, v.w);
            *reinterpret_cast<float4*>(ps + 4 * LPR * k) = v;
        }
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            const float m2 = __shfl_xor_sync(0xffffffffu, lse_m, o);
            const float s2v = __shfl_xor_sync(0xffffffffu, lse_s, o);
            lse2_merge(lse_m, lse_s, m2, s2v);
        }
        if (l == 0) {
            float2* pj = reinterpret_cast<float2*>(a.Jpart) + (size_t)blockIdx.y * a.bl_pad + row;
            *pj = make_float2(lse_m, lse_s);
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// backward: lanes span the dims, a warp owns RI rows, 8 warps per CTA; the two column sums of a warp
// are staged per JS columns and reduced by the CTA, then added to the global accumulators.
// ------------------------------------------------------------------------------------------------------
template <int DPT> struct CvBwdGeom {
    static constexpr int VEC = DPT < 4 ? DPT : 4;
    static constexpr int NCH = DPT / VEC;
    static constexpr int DP = 32 * DPT;
    static constexpr int CH = 32 * VEC;
    static constexpr int JT = CvGeom<DPT>::JT;
    static constexpr int JS = (512 / DP) < 1 ? 1 : ((512 / DP) > JT ? JT : (512 / DP));   // columns per staging buffer
};

template <int DPT, int RI>
__global__ void __launch_bounds__(kBwdWarps * 32, colvar_bwd_res(DPT))
tc_bwd_colvar_kernel(const BwdFusedArgs a) {
    using GEO = CvBwdGeom<DPT>;
    constexpr int VEC = GEO::VEC, NCH = GEO::NCH, DP = GEO::DP, CH = GEO::CH, JT = GEO::JT, JS = GEO::JS;
    constexpr int TILE = JT * 3 * DP;
    constexpr int ROWS = kBwdWarps * RI;
    constexpr int GST = kBwdWarps * JS * 2 * DP;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* col_tiles = reinterpret_cast<float*>(smem_raw);                   // [kStages][TILE]
    float* s2_tiles = col_tiles + (size_t)kStages * TILE;                    // [kStages][ROWS][JT]
    float* gq_buf = s2_tiles + (size_t)kStages * ROWS * JT;                  // [kBwdWarps][RI][JT]
    float* gstage = gq_buf + (size_t)kBwdWarps * RI * JT;                    // [kBwdWarps][JS][2][DP]
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(gstage + (size_t)GST);
    uint64_t* bar_empty = bar_full + kStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row0 = blockIdx.x * ROWS + warp * RI;

    float zr[RI][DPT], gps[RI][DPT], A[RI][DPT];
#pragma unroll
    for (int r = 0; r < RI; ++r) {
        const bool valid = (row0 + r) < a.bl_pad;
        const size_t base = (size_t)min(row0 + r, a.bl_pad - 1) * DP;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                const int dd = c * CH + VEC * lane + e;
                zr[r][c * VEC + e] = a.zs[base + dd];
                gps[r][c * VEC + e] = valid ? a.gps[base + dd] : 0.0f;
                A[r][c * VEC + e] = 0.0f;
            }
        }
    }

    const int j0 = blockIdx.y * a.js_len;
    const int j1 = min(a.bg_pad, j0 + a.js_len);
    const int ntiles = (j1 - j0) / JT;
    constexpr uint32_t kTxBytes = (TILE + ROWS * JT) * sizeof(float);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], kBwdWarps); }
        mbar_fence_init();
    }
    __syncthreads();

    auto issue = [&](int t) {
        const int sn = t % kStages;
        if (lane == 0) {
            if (t >= kStages) mbar_wait(&bar_empty[sn], ((t / kStages) - 1) & 1);
            mbar_arrive_expect_tx(&bar_full[sn], kTxBytes);
            bulk_g2s(col_tiles + (size_t)sn * TILE, a.mu_pad + (size_t)(j0 + t * JT) * 3 * DP, TILE * sizeof(float), &bar_full[sn]);
        }
        __syncwarp();
        for (int r = lane; r < ROWS; r += 32)
            bulk_g2s(s2_tiles + ((size_t)sn * ROWS + r) * JT,
                     a.s2 + (size_t)min((int)(blockIdx.x * ROWS + r), a.bl_pad - 1) * a.ld_s2 + (j0 + t * JT), JT * sizeof(float), &bar_full[sn]);
    };
    if (warp == 0 && ntiles > 0) issue(0);

    float* gq = gq_buf + (size_t)warp * RI * JT;
    for (int t = 0; t < ntiles; ++t) {
        const int st = t % kStages;
        if (warp == 0 && t + 1 < ntiles) issue(t + 1);
        mbar_wait(&bar_full[st], (t / kStages) & 1);
        const float* tile = col_tiles + (size_t)st * TILE;
        const float* s2t = s2_tiles + ((size_t)st * ROWS + warp * RI) * JT;
        const int jt0 = j0 + t * JT;
        const bool special = (a.w.mss && jt0 == 0) || (jt0 + JT > a.w.b_glob);

        __syncwarp();
        for (int idx = lane; idx < RI * JT; idx += 32) {
            const int r = idx / JT, jj = idx % JT;
            const int row = row0 + r;
            float rho = 1.0f, l2 = 0.0f;
            if (special) weight_of(a.w, a.row_offset + row, jt0 + jj, rho, l2);
            const int rowc = min(row, a.bl_pad - 1);
            const float qv = ex2(l2 - s2t[idx] - __ldg(a.J2 + rowc));
            gq[idx] = (jt0 + jj < a.w.b_glob && row < a.b_loc) ? __ldg(a.gj + rowc) * qv : 0.0f;
        }
        __syncwarp();

        for (int sub = 0; sub < JT; sub += JS) {
            float* gst = gstage + (size_t)warp * JS * 2 * DP;
            for (int u = 0; u < JS; ++u) {
                const int jj = sub + u;
                float sj[DPT], nm[DPT], c2[DPT], Gmu[DPT], Glv[DPT];
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        const int dd = c * CH + VEC * lane + e;
                        sj[c * VEC + e] = tile[(size_t)jj * 3 * DP + dd];
                        nm[c * VEC + e] = tile[(size_t)jj * 3 * DP + DP + dd];
                        c2[c * VEC + e] = tile[(size_t)jj * 3 * DP + 2 * DP + dd];
                        Gmu[c * VEC + e] = 0.0f; Glv[c * VEC + e] = 0.0f;
                    }
                }
#pragma unroll
                for (int r = 0; r < RI; ++r) {
                    float rho = 1.0f, l2 = 0.0f;
                    if (special) weight_of(a.w, a.row_offset + row0 + r, jt0 + jj, rho, l2);
                    const float g = gq[r * JT + jj];
#pragma unroll
                    for (int e = 0; e < DPT; ++e) {
                        const float dl = fmaf(zr[r][e], sj[e], nm[e]);
                        const float q = dl * dl;
                        const float tt = c2[e] - q;
                        float ev = ex2(tt);                            // no clamp needed: a clamped pair is masked below
                        if (special) ev *= rho;
                        const float coef = fmaf(ev, gps[r][e], g);
                        const float rr = (tt < -kK50) ? 0.0f : coef;
                        const float wv = rr * dl;
                        A[r][e] = fmaf(wv, sj[e], A[r][e]);
                        Gmu[e] += wv;
                        Glv[e] = fmaf(rr, fmaf(q, kLn2, -0.5f), Glv[e]);
                    }
                }
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        const int dd = c * CH + VEC * lane + e;
                        gst[(size_t)u * 2 * DP + dd] = Gmu[c * VEC + e];
                        gst[(size_t)u * 2 * DP + DP + dd] = Glv[c * VEC + e];
                    }
                }
            }
            __syncthreads();
            for (int f = threadIdx.x; f < JS * 2 * DP / 4; f += kBwdWarps * 32) {
                const int col = f / (2 * DP / 4), chunk = f % (2 * DP / 4);       // chunk < DP/4: mu part, else logvar part
                float4 acc = *reinterpret_cast<const float4*>(gstage + (size_t)col * 2 * DP + 4 * chunk);
#pragma unroll
                for (int w = 1; w < kBwdWarps; ++w) {
                    const float4 v = *reinterpret_cast<const float4*>(gstage + ((size_t)w * JS + col) * 2 * DP + 4 * chunk);
                    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                }
                const bool is_mu = chunk < DP / 4;
                float* dst = (is_mu ? a.Gacc : a.Gacc2) + (size_t)(jt0 + sub + col) * DP + 4 * (is_mu ? chunk : chunk - DP / 4);
                red_add_v4_cv(dst, acc.x, acc.y, acc.z, acc.w);
            }
            __syncthreads();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_empty[st]);
    }

#pragma unroll
    for (int r = 0; r < RI; ++r) {
        if (row0 + r >= a.bl_pad) continue;
        const size_t base = ((size_t)blockIdx.y * a.bl_pad + row0 + r) * DP;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) a.Apart[base + c * CH + VEC * lane + e] = A[r][c * VEC + e];
        }
    }
}

// With the decomposition (a.gc != nullptr) the row-local densities of solvers/tc.py:107,112 add their gradients, the terms of
// rowdensity_bwd_kernel: condx_i = sum_d lp(z_id; mu_rd, lv_rd) to grad_z[i] and to row r = row_offset + i of grad_mu / grad_lv
// (the thread that owns (r, d) of the column part adds them, so no two threads write one element), pz_i = sum_d lp(z_id; 0, 0)
// to grad_z[i].
// Peer exchange (a.scratch_parts != nullptr): after the barrier that says every rank's sweep is done, the column part covers this
// rank's rows only; their mu and logvar column sums are added up over all ranks' scratch in rank order (the reduce-scatter is this
// kernel's load phase), and mu_all / lv / grad_mu / grad_lv are this rank's rows at local indices.
// Fused reparameterize (a.eps != nullptr, z = mu + eps * exp(lv / 2) of the local rows): the thread of local element (i, d) writes
// grad_z[i] and also row r = row_offset + i of grad_mu / grad_lv with its own grad_z chained through z (as rows_own_mu does in
// bwd_fused_finalize_kernel), so no thread reads another's output; the column part then skips the local rows.
__global__ void bwd_colvar_finalize_kernel(const BwdFinArgs a, const float* __restrict__ colpack, const float* __restrict__ Glv) {
    const bool peer = a.scratch_parts != nullptr;
    const bool rows_own = a.eps != nullptr;
    if (peer && a.sync.on()) peer_barrier(a.sync);
    const int64_t n_row = (int64_t)a.b_loc * a.d;
    const int64_t n_col = (int64_t)(peer ? a.b_loc : a.b_glob) * a.d;
    const int64_t mrow0 = peer ? 0 : a.row_offset;                    // row of mu_all / lv that holds local row 0
    const size_t glv_off = a.g_off + (size_t)a.bg_pad * a.dp * sizeof(float);    // Glv follows Gpart in every rank's scratch
    // gradients of mu / logvar at global row j (column sums, plus the condx terms of a local row)
    auto col_grad = [&](int j, int dd, float& gmu, float& glv) {
        const size_t o = (size_t)j * a.dp + dd;
        const float sj = colpack[(size_t)j * 3 * a.dp + dd];
        float gm, gl;
        if (peer) {
            gm = 0.0f; gl = 0.0f;
            for (int p0 = 0; p0 < a.n_ranks; p0 += 4) {
                float vm[4], vl[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const char* base = static_cast<const char*>(a.scratch_parts[p0 + q < a.n_ranks ? p0 + q : p0]);
                    vm[q] = *reinterpret_cast<const volatile float*>(base + a.g_off + o * sizeof(float));
                    vl[q] = *reinterpret_cast<const volatile float*>(base + glv_off + o * sizeof(float));
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (p0 + q < a.n_ranks) { gm += vm[q]; gl += vl[q]; }
                }
            }
        } else {
            gm = a.Gpart[o]; gl = Glv[o];
        }
        gmu = kTwoLn2 * sj * gm; glv = gl;
        const int i = j - a.row_offset;
        if (a.gc != nullptr && i >= 0 && i < a.b_loc) {
            const float m = a.mu_all[(mrow0 + i) * a.ldmu + dd], l = a.lv[(mrow0 + i) * a.ldlv + dd];
            float t, iv;
            const float lp = lp_unfloored(a.z[(int64_t)i * a.ldz + dd], m, l, t, iv);
            const float gc = lp_passes_grad(lp) ? a.gc[i] : 0.0f;
            gmu += gc * t * iv;
            glv += gc * 0.5f * (t * t * iv - 1.0f);
        }
    };
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_row + n_col; idx += (int64_t)gridDim.x * blockDim.x) {
        if (idx < n_row) {
            const int i = (int)(idx / a.d), dd = (int)(idx % a.d);
            const size_t o = (size_t)i * a.dp + dd;
            float sa = 0.0f;
            for (int s = 0; s < a.n_js; ++s) sa += a.Apart[(size_t)s * a.bl_pad * a.dp + o];
            float gz = -kTwoLn2 * sa;
            if (a.gc != nullptr) {
                const int64_t r = mrow0 + i;
                const float x = a.z[(int64_t)i * a.ldz + dd];
                float t, iv, t0, iv0;
                const float lp = lp_unfloored(x, a.mu_all[r * a.ldmu + dd], a.lv[r * a.ldlv + dd], t, iv);
                const float lp0 = lp_unfloored(x, 0.0f, 0.0f, t0, iv0);
                const float gc = lp_passes_grad(lp) ? a.gc[i] : 0.0f, gp = lp_passes_grad(lp0) ? a.gpz[i] : 0.0f;
                gz += -gc * t * iv + -gp * t0 * iv0;
            }
            a.grad_z[(int64_t)i * a.ldgz + dd] = gz;
            if (rows_own) {                                           // through z = mu + eps * std
                float gmu, glv;
                col_grad(a.row_offset + i, dd, gmu, glv);
                const float lv = a.lv[(mrow0 + i) * a.ldlv + dd];
                gmu += gz;
                glv += gz * a.eps[(int64_t)i * a.ldeps + dd] * (0.5f * expf(0.5f * lv));
                const int64_t grow = peer ? i : a.row_offset + i;
                a.grad_mu[grow * a.ldgmu + dd] = gmu;
                a.grad_lv[grow * a.ldglv + dd] = glv;
            }
        } else {
            const int64_t k = idx - n_row;
            const int j = (int)(k / a.d) + (peer ? a.row_offset : 0), dd = (int)(k % a.d);
            const int i = j - a.row_offset;
            if (rows_own && i >= 0 && i < a.b_loc) continue;          // written by the row part
            float gmu, glv;
            col_grad(j, dd, gmu, glv);
            const int64_t grow = peer ? i : j;                        // grad_mu / grad_lv: this rank's rows only in the peer mode
            a.grad_mu[grow * a.ldgmu + dd] = gmu;
            a.grad_lv[grow * a.ldglv + dd] = glv;
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------------
cudaError_t launch_colvar_prep(const ColPrepArgs& a, cudaStream_t st) {
    // the ranks' published buffers are dense, 16-byte aligned allocations: 16-byte gathers when the row pitch keeps them aligned
    const bool vec = a.mu_parts != nullptr && a.d % 4 == 0 && a.ld_part % 4 == 0;
    const int64_t n = (int64_t)(a.bg_pad + a.bl_pad) * a.dp;
    int64_t g = (n + 255) / 256; if (g > 148 * 16) g = 148 * 16;
    LaunchScope scope(kKernNone, st);
    if (a.mu_parts == nullptr) colvar_prep_kernel<false, 1><<<(int)g, 256, 0, st>>>(a);
    else if (vec)              colvar_prep_kernel<true, 4><<<(int)g, 256, 0, st>>>(a);
    else                       colvar_prep_kernel<true, 1><<<(int)g, 256, 0, st>>>(a);
    return cudaGetLastError();
}

template <int LPR>
static cudaError_t launch_fwd_colvar_t(const Plan& p, const FwdArgs& a, cudaStream_t st) {
    constexpr auto kern = tc_fwd_colvar_kernel<LPR>;
    const size_t smem = (size_t)kStages * CvGeom<LPR>::TILE * sizeof(float) + 2 * kStages * sizeof(uint64_t);
    if (cudaError_t e = allow_dynamic_smem<kern>(smem)) return e;
    LaunchScope scope(kKernFwd, st);
    kern<<<dim3(p.n_rb_fwd, p.n_js_fwd), kFwdWarps * 32, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_fwd_colvar(const Plan& p, const FwdArgs& a, cudaStream_t st) {
    switch (p.dpt) {
        case 1:  return launch_fwd_colvar_t<1>(p, a, st);
        case 2:  return launch_fwd_colvar_t<2>(p, a, st);
        case 4:  return launch_fwd_colvar_t<4>(p, a, st);
        case 8:  return launch_fwd_colvar_t<8>(p, a, st);
        case 16: return launch_fwd_colvar_t<16>(p, a, st);
        default: return cudaErrorInvalidValue;
    }
}

template <int DPT>
static cudaError_t launch_bwd_colvar_t(const Plan& p, const BwdFusedArgs& a, cudaStream_t st) {
    using GEO = CvBwdGeom<DPT>;
    constexpr int RI = colvar_bwd_rows_per_warp(DPT), ROWS = kBwdWarps * RI;
    constexpr auto kern = tc_bwd_colvar_kernel<DPT, RI>;
    const size_t smem = ((size_t)kStages * GEO::JT * 3 * GEO::DP + (size_t)kStages * ROWS * GEO::JT + (size_t)kBwdWarps * RI * GEO::JT
                         + (size_t)kBwdWarps * GEO::JS * 2 * GEO::DP) * sizeof(float) + 2 * kStages * sizeof(uint64_t);
    if (cudaError_t e = allow_dynamic_smem<kern>(smem)) return e;
    LaunchScope scope(kKernBwdRow, st);
    kern<<<dim3(p.n_rb_bwd, p.n_js_bwd), kBwdWarps * 32, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_bwd_colvar(const Plan& p, const BwdFusedArgs& a, cudaStream_t st) {
    switch (p.dpt) {
        case 1:  return launch_bwd_colvar_t<1>(p, a, st);
        case 2:  return launch_bwd_colvar_t<2>(p, a, st);
        case 4:  return launch_bwd_colvar_t<4>(p, a, st);
        case 8:  return launch_bwd_colvar_t<8>(p, a, st);
        case 16: return launch_bwd_colvar_t<16>(p, a, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_bwd_colvar_finalize(const Plan& p, const BwdFinArgs& a, const float* colpack, const float* Glv, cudaStream_t st) {
    const int64_t n = (int64_t)p.b_loc * p.d + (int64_t)(a.scratch_parts != nullptr ? p.b_loc : p.b_glob) * p.d;
    int64_t g = (n + 255) / 256; if (g > 148 * 16) g = 148 * 16; if (g < 1) g = 1;
    LaunchScope scope(kKernNone, st);
    bwd_colvar_finalize_kernel<<<(int)g, 256, 0, st>>>(a, colpack, Glv);
    return cudaGetLastError();
}

}  // namespace tcelbo
