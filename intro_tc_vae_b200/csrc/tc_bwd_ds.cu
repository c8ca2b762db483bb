// Fused backward sweep of the TC-ELBO estimator (sm_100a): ONE recomputation of e_ijd = 2^-qc per log-density yields all
// three gradients of ops.py:80-115's autograd graph:
//     r_ijd  = (gJ_i q_ij + gP_i rho_ij e_ijd / S_id) * [q_ijd <= qmax_id]      (mask of the -50 clamp)
//     A_id   = sum_j r dl             -> grad_z        (row-local, registers)
//     CR_id  = sum_j r (2 ln2 qc - 1) -> grad_logvar   (row-local, registers)
//     G_jd   = sum_i r dl ns_id       -> grad_mu       (column sum over rows)
// The exponent is carried shifted, q' = dl^2 - 1/(2 ln2) (one FFMA2), so that 2 ln2 qc - 1 = 2 ln2 qc' and the logvar sum is a
// plain sum_j r qc'; 2^-qc' = e * exp(1/2) and the exp(-1/2) is folded into the per-row coefficient gP/S.
//
// Mapping ("dims across warps"):
//   * a lane owns ONE latent dim; the CH warps of a row group cover a 32*CH-dim slice (CH = 4 at D >= 128), and every warp
//     of the group holds the same 2*RP rows.  The two halves of a packed f32x2 register are two ROWS of that dim, so the
//     column operand mu_jd is one scalar broadcast into both halves (FFMA2's .F32 operand form) and the per-(i,j) joint
//     coefficients come out of shared memory already paired.
//   * the column gradient of a warp's rows therefore accumulates in ONE register per column and goes straight to the
//     global accumulator with a coalesced 128-byte red.global.add.f32 -- no shared-memory staging, no cross-warp
//     reduction, no mbarrier hand-off between the warps of a CTA (the rows-across-warps kernel of round 1 spent 13-15 % of
//     its warp time in that hand-off, profiles/r1_bwd_variant_sweep.md; it is gone, profiles/r2_bwd_ds_sweep.md).  Warps meet
//     only at the TMA pipeline's barriers.
//   * both tile operands arrive by tensor-map TMA (cp.async.bulk.tensor.2d -> UTMALDG): a [JT x 32*CH] box of the padded
//     column operand and a [ROWS x JT] box of the saved joint exponents s2 (rows past the padded batch are zero-filled by
//     the TMA unit instead of clamped in software).
//   * D = 256 / 512 walk 128-dim slices: row-local and column sums are independent per dim, only the joint coefficients
//     are shared, so a slice is a self-contained sweep (blocks = (slice, row block), balanced segments as in the forward).
#include <cuda.h>

#include "tc_common.cuh"
#include "tc_instr.h"
#include "tc_kernels.h"

namespace tcelbo {

struct alignas(64) BwdDsArgs {
    CUtensorMap map_mu;                                                      // [bg_pad][pitch] fp32, box [JT][32*CH]
    CUtensorMap map_s2;                                                      // [bl_pad][ld_s2] fp32, box [ROWS][JT]
    const float* zs; const float* ns; const float* qmax; const float* gps;   // [bl_pad][pitch]
    const float* gj; const float* J2;                                        // [bl_pad]
    float* Apart; float* CRpart;                                             // [slots][bl_pad][pitch]
    float* Gacc;                                                             // [bg_pad][pitch], zeroed by the caller
    int b_loc, bl_pad, bg_pad, row_offset, pitch;
    Segments seg; int n_rb;
    Weights w;
};

__device__ __forceinline__ void red_add_f32(float* addr, float v) {
    asm volatile("red.global.add.f32 [%0], %1;" :: "l"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// One column for this warp's RP row pairs (this lane's dim).  kSpecial: the tile holds a stratified or a padding column.
template <int RP, bool kSpecial>
__device__ __forceinline__ float ds_column(float mu, const float* __restrict__ gq_col, int i_glob0, int j, const Weights& w,
                                           const u64 (&zs2)[RP], const u64 (&ns2)[RP], const float (&qmx)[2 * RP],
                                           const u64 (&gps2)[RP], u64 (&A2)[RP], u64 (&CR2)[RP]) {
    const u64 mu2 = pack2(mu, mu);
    const u64 nk2 = pack2(-kInvTwoLn2, -kInvTwoLn2);
    u64 Ga = 0ull, Gb = 0ull;
#pragma unroll
    for (int p = 0; p < RP; ++p) {
        const u64 gq2 = *reinterpret_cast<const u64*>(gq_col + 2 * p);                    // (gJ q)_(2p, j), (gJ q)_(2p+1, j)
        const u64 dl2 = ffma2(mu2, ns2[p], zs2[p]);
        const u64 q2 = ffma2(dl2, dl2, nk2);                                               // q' = q - 1/(2 ln2)
        float q0, q1;
        unpack2(q2, q0, q1);
        // A clamped pair contributes r = 0 whatever its weight, so the exponent needs no min(q, qmax) here (the forward's clamp
        // decides the VALUE of a clamped term; the backward only needs to know that it was clamped): 2 ALU instructions less
        // per pair of log-densities, 3.42 -> 3.11 ms at 8192 x 8192 x 128.
        u64 e2 = pack2(ex2(-q0), ex2(-q1));
        if (kSpecial) {
            float r0, r1, l2;
            weight_of(w, i_glob0 + 2 * p, j, r0, l2);
            weight_of(w, i_glob0 + 2 * p + 1, j, r1, l2);
            e2 = fmul2(e2, pack2(r0, r1));
        }
        const u64 coef2 = ffma2(e2, gps2[p], gq2);
        float k0, k1;                                // clamp mask as FSETP + FSEL on the ALU pipe (a NaN q gives r = 0, like torch.clamp's backward)
        unpack2(coef2, k0, k1);
        const u64 r2 = pack2(q0 <= qmx[2 * p] ? k0 : 0.0f, q1 <= qmx[2 * p + 1] ? k1 : 0.0f);
        const u64 t2 = fmul2(r2, dl2);
        A2[p] = fadd2(A2[p], t2);
        CR2[p] = ffma2(r2, q2, CR2[p]);
        if (p & 1) Gb = ffma2(t2, ns2[p], Gb); else Ga = ffma2(t2, ns2[p], Ga);
    }
    float lo, hi;
    unpack2(fadd2(Ga, Gb), lo, hi);
    return lo + hi;
}

template <int RP, int CH, int NW, int MINB, int JT>
__global__ void __launch_bounds__(NW * 32, MINB)
tc_bwd_ds_kernel(const __grid_constant__ BwdDsArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    constexpr int RW = 2 * RP;                                               // rows per warp
    constexpr int NRG = NW / CH;                                             // row groups per CTA
    constexpr int ROWS = NRG * RW;
    constexpr int DPS = 32 * CH;                                             // dims per slice
    constexpr int TILE = JT * DPS;
    static_assert(NW % CH == 0, "warps must split into whole row groups");
    static_assert((TILE * 4) % 128 == 0 && (ROWS * JT * 4) % 128 == 0, "TMA destinations must stay 128-byte aligned");

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* mu_tiles = reinterpret_cast<float*>(smem_raw);                    // [kStages][JT][DPS]
    float* s2_tiles = mu_tiles + (size_t)kStages * TILE;                     // [kStages][ROWS][JT]
    float* gq_buf = s2_tiles + (size_t)kStages * ROWS * JT;                  // [NW][JT][RW]   (private per warp)
    float* rowc = gq_buf + (size_t)NW * JT * RW;                             // [NW][RW][2]    gJ_i, -J2_i of the warp's rows
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(rowc + (size_t)NW * RW * 2);
    uint64_t* bar_empty = bar_full + kStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunk = warp % CH, rgrp = warp / CH;
    const int pitch = a.pitch;
    const int T = a.bg_pad / JT;
    // same balanced-segment plan as the other sweeps: blocks = (slice, row block), linearised block-major (tc_layout.h)
    const int64_t g_begin = seg_begin(a.seg, blockIdx.x);
    const int ntiles = seg_len(a.seg, blockIdx.x);
    int q = (int)(g_begin / T);
    const int t_first = (int)(g_begin - (int64_t)q * T);
    int rb0 = (q % a.n_rb) * ROWS;
    int row0 = rb0 + rgrp * RW;
    int d0 = (q / a.n_rb) * DPS;
    int dl_ = d0 + chunk * 32 + lane;                                        // this lane's dim

    u64 zs2[RP], ns2[RP], gps2[RP], A2[RP], CR2[RP];
    float qmx[2 * RP];
    float* my_rowc = rowc + (size_t)warp * RW * 2;
    auto load_rows = [&]() {
#pragma unroll
        for (int p = 0; p < RP; ++p) {
            float vz[2], vn[2], vq[2], vg[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int row = row0 + 2 * p + h;
                const bool valid = row < a.bl_pad;
                const size_t o = (size_t)min(row, a.bl_pad - 1) * pitch + dl_;
                vz[h] = __ldg(a.zs + o); vn[h] = __ldg(a.ns + o);
                vq[h] = __ldg(a.qmax + o) - kInvTwoLn2;                      // the sweep compares q' = q - 1/(2 ln2)
                vg[h] = valid ? __ldg(a.gps + o) * kRsqrtE : 0.0f;           // 2^-q' = 2^-q * exp(1/2): exp(-1/2) folded in here
            }
            zs2[p] = pack2(vz[0], vz[1]); ns2[p] = pack2(vn[0], vn[1]); gps2[p] = pack2(vg[0], vg[1]);
            qmx[2 * p] = vq[0]; qmx[2 * p + 1] = vq[1];
            A2[p] = 0ull; CR2[p] = 0ull;
        }
        __syncwarp();
        if (lane < RW) {
            const int row = row0 + lane;
            const bool valid = row < a.b_loc;
            const int rc = min(row, a.bl_pad - 1);
            // rows past the batch: coefficient 0 * 2^(-inf) = 0 (their J2 is not written, and the s2 of rows past the padded batch
            // is TMA zero fill: 2^(-J2 - 0) alone would overflow to inf for wide latents and 0 * inf poison the column sums)
            my_rowc[2 * lane] = valid ? __ldg(a.gj + rc) : 0.0f;
            my_rowc[2 * lane + 1] = valid ? -__ldg(a.J2 + rc) : -1.0e30f;
        }
        __syncwarp();
    };
    auto flush_rows = [&]() {
        const int slot = (int)blockIdx.x - seg_of(a.seg, (int64_t)q * T);
#pragma unroll
        for (int p = 0; p < RP; ++p) {
            float al, ah, cl, ch;
            unpack2(A2[p], al, ah); unpack2(CR2[p], cl, ch);
            const int row = row0 + 2 * p;
            const size_t o = ((size_t)slot * a.bl_pad + row) * pitch + dl_;
            if (row < a.bl_pad) { a.Apart[o] = al; a.CRpart[o] = cl; }
            if (row + 1 < a.bl_pad) { a.Apart[o + pitch] = ah; a.CRpart[o + pitch] = ch; }
        }
    };
    load_rows();

    constexpr uint32_t kTxBytes = (TILE + ROWS * JT) * sizeof(float);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], NW); }
        mbar_fence_init();
    }
    __syncthreads();

    auto issue = [&](int t, int tn, int rbn, int dn) {                       // one elected thread
        const int sn = t % kStages;
        if (t >= kStages) mbar_wait(&bar_empty[sn], ((t / kStages) - 1) & 1);
        mbar_arrive_expect_tx(&bar_full[sn], kTxBytes);
        tma_load_2d(mu_tiles + (size_t)sn * TILE, &a.map_mu, dn, tn * JT, &bar_full[sn]);
        tma_load_2d(s2_tiles + (size_t)sn * ROWS * JT, &a.map_s2, tn * JT, rbn, &bar_full[sn]);
    };
    if (threadIdx.x == 0 && ntiles > 0) issue(0, t_first, rb0, d0);

    float* gq = gq_buf + (size_t)warp * JT * RW;
    int t_in = t_first;
    for (int t = 0; t < ntiles; ++t, ++t_in) {
        if (t_in == T) {                                                     // segment crosses into the next block
            flush_rows();
            ++q; t_in = 0;
            rb0 = (q % a.n_rb) * ROWS; row0 = rb0 + rgrp * RW; d0 = (q / a.n_rb) * DPS; dl_ = d0 + chunk * 32 + lane;
            load_rows();
        }
        const int st = t % kStages;
        if (threadIdx.x == 0 && t + 1 < ntiles) {
            int tn = t_in + 1, rbn = rb0, dn = d0;
            if (tn == T) { tn = 0; rbn = ((q + 1) % a.n_rb) * ROWS; dn = ((q + 1) / a.n_rb) * DPS; }
            issue(t + 1, tn, rbn, dn);
        }
        mbar_wait(&bar_full[st], (t / kStages) & 1);
        const float* tile = mu_tiles + (size_t)st * TILE + chunk * 32 + lane;
        const float* s2t = s2_tiles + ((size_t)st * ROWS + rgrp * RW) * JT;
        const int jt0 = t_in * JT;
        const bool special = (a.w.mss && jt0 == 0) || (jt0 + JT > a.w.b_glob);

        // joint-term coefficients gJ_i q_ij of this warp's rows, transposed to [column][row] so that a column's RW values are
        // RP ready-made f32x2 pairs (one broadcast LDS.64 each in the sweep).  Value idx = lane + 32 k covers row lane/JT + RPI k
        // and column lane % JT: every address is a per-lane base plus a compile-time offset.
        __syncwarp();
        {
            constexpr int RPI = 32 / JT;                                     // rows per iteration
            const int jj = lane % JT, rl = lane / JT;
            const float* s2p = s2t + lane;
            const float* rcp = my_rowc + 2 * rl;
            float* gqp = gq + jj * RW + rl;
            if (special) {
#pragma unroll
                for (int k = 0; k < RW / RPI; ++k) {
                    float rho, l2;
                    weight_of(a.w, a.row_offset + row0 + rl + RPI * k, jt0 + jj, rho, l2);
                    const float2 c = *reinterpret_cast<const float2*>(rcp + 2 * RPI * k);
                    const float qv = ex2(l2 - s2p[32 * k] + c.y);
                    gqp[RPI * k] = (jt0 + jj < a.w.b_glob) ? c.x * qv : 0.0f;
                }
            } else {
#pragma unroll
                for (int k = 0; k < RW / RPI; ++k) {
                    const float2 c = *reinterpret_cast<const float2*>(rcp + 2 * RPI * k);   // (gJ_i, -J2_i)
                    gqp[RPI * k] = c.x * ex2(c.y - s2p[32 * k]);
                }
            }
        }
        __syncwarp();

        float* gptr = a.Gacc + (size_t)jt0 * pitch + dl_;                   // running pointer: one 64-bit add per column
        if (special) {
#pragma unroll 2
            for (int jj = 0; jj < JT; ++jj) {
                const float g = ds_column<RP, true>(tile[jj * DPS], gq + jj * RW, a.row_offset + row0, jt0 + jj, a.w, zs2, ns2, qmx, gps2, A2, CR2);
                red_add_f32(gptr, g);
                gptr += pitch;
            }
        } else {
#pragma unroll 8
            for (int jj = 0; jj < JT; ++jj) {
                const float g = ds_column<RP, false>(tile[jj * DPS], gq + jj * RW, 0, 0, a.w, zs2, ns2, qmx, gps2, A2, CR2);
                red_add_f32(gptr, g);
                gptr += pitch;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_empty[st]);
    }
    flush_rows();
}

// ------------------------------------------------------------------------------------------------------
// launch
// ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D fp32 tensor map: `rows` x `cols` elements with a row pitch of `ld` elements, box `box_rows` x `box_cols`, zero fill
static bool make_map_2d(CUtensorMap* m, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * sizeof(float)};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int K>
static cudaError_t launch_bwd_ds_t(const Plan& p, const BwdFusedArgs& u, cudaStream_t st) {
    constexpr BwdDsConfig c = kBwdDsConfigs[K];
    constexpr int RP = c.rp, CH = c.ch, NW = c.nw, JT = c.jt, ROWS = (NW / CH) * 2 * RP, DPS = 32 * CH;
    constexpr auto kern = tc_bwd_ds_kernel<RP, CH, NW, c.minb, JT>;
    const size_t smem = ((size_t)kStages * JT * DPS + (size_t)kStages * ROWS * JT + (size_t)NW * JT * 2 * RP + (size_t)NW * 2 * RP * 2) * sizeof(float)
                        + 2 * kStages * sizeof(uint64_t);
    if (cudaError_t e = allow_dynamic_smem<kern>(smem)) return e;
    BwdDsArgs a;
    if (!make_map_2d(&a.map_mu, u.mu_pad, (uint64_t)p.bg_pad, (uint64_t)p.dp, (uint64_t)p.dp, JT, DPS)) return cudaErrorNotSupported;
    if (!make_map_2d(&a.map_s2, u.s2, (uint64_t)p.bl_pad, (uint64_t)p.bg_pad, (uint64_t)u.ld_s2, ROWS, JT)) return cudaErrorNotSupported;
    a.zs = u.zs; a.ns = u.ns; a.qmax = u.qmax; a.gps = u.gps; a.gj = u.gj; a.J2 = u.J2;
    a.Apart = u.Apart; a.CRpart = u.CRpart; a.Gacc = u.Gacc;
    a.b_loc = u.b_loc; a.bl_pad = u.bl_pad; a.bg_pad = u.bg_pad; a.row_offset = u.row_offset; a.pitch = p.dp;
    a.seg = p.seg_bwd; a.n_rb = p.n_rb_bwd; a.w = u.w;
    LaunchScope scope(kKernBwdRow, st);
    return launch_pdl(kern, dim3(p.seg_bwd.n_ctas), dim3(NW * 32), smem, st, a);
}

// Elementwise over [B,D]: sum the column-split partials of the row-local sums (8 independent loads in flight), scale,
// and add the fused KL gradient when asked (ops.py:161-163).
__global__ void bwd_fused_finalize_kernel(const BwdFinArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int64_t n_row = (int64_t)a.b_loc * a.d;
    const int64_t n_col = a.scratch_parts != nullptr ? 0 : (int64_t)a.b_glob * a.d;
    const size_t split_stride = (size_t)a.bl_pad * a.dp;
    const bool rows_own_mu = a.scratch_parts != nullptr || a.eps != nullptr;   // the row threads also write grad_mu of the local rows
    if (a.scratch_parts != nullptr && a.sync.on()) peer_barrier(a.sync);        // every rank's sweep has finished: their column sums are final
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_row + n_col; idx += (int64_t)gridDim.x * blockDim.x) {
        if (idx < n_row) {
            const int i = (int)(idx / a.d), dd = (int)(idx % a.d);
            const size_t o = (size_t)i * a.dp + dd;
            float sa = 0.0f, sc = 0.0f;
            // partial slots of this (slice, row block): one per segment that touches the block
            const int64_t qb = (int64_t)(dd / a.slice_dp) * a.n_rb + i / a.rows_per_block;
            const int n_slots = seg_slots(a.seg, qb, a.tiles_per_block);
            for (int s0 = 0; s0 < n_slots; s0 += 4) {
                float va[4], vc[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool ok = s0 + k < n_slots;
                    va[k] = ok ? __ldg(a.Apart + (size_t)(s0 + k) * split_stride + o) : 0.0f;
                    vc[k] = ok ? __ldg(a.CRpart + (size_t)(s0 + k) * split_stride + o) : 0.0f;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) { sa += va[k]; sc += vc[k]; }
            }
            float glv = a.vr[o] * (kTwoLn2 * sc);                         // the sweep accumulates sum r (c - 1/(2 ln2))
            const float lv = (a.gk != nullptr || a.eps != nullptr) ? a.lv[(int64_t)i * a.ldlv + dd] : 0.0f;
            if (a.gk != nullptr) glv += a.gk[i] * 0.5f * (expf(lv) - 1.0f);
            const float gz = kTwoLn2 * a.ns[o] * sa;
            if (a.eps != nullptr) glv += gz * a.eps[(int64_t)i * a.ldeps + dd] * (0.5f * expf(0.5f * lv));    // through z = mu + eps*std
            a.grad_z[(int64_t)i * a.ldgz + dd] = gz;
            a.grad_lv[(int64_t)i * a.ldglv + dd] = glv;
            if (rows_own_mu) {
                const size_t og = (size_t)(a.row_offset + i) * a.dp + dd;
                float g = 0.0f;
                if (a.scratch_parts != nullptr) {
                    // reduce-scatter of the column gradient as this kernel's load phase: the local rows of every rank's accumulator
                    for (int p0 = 0; p0 < a.n_ranks; p0 += 8) {
                        float v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            v[k] = (p0 + k < a.n_ranks)
                                       ? *reinterpret_cast<const volatile float*>(static_cast<const char*>(a.scratch_parts[p0 + k]) + a.g_off + og * sizeof(float))
                                       : 0.0f;
#pragma unroll
                        for (int k = 0; k < 8; ++k) g += v[k];
                    }
                } else {
                    g = a.Gpart[og];
                }
                g *= -kTwoLn2;
                // mu_all holds this rank's rows only in the peer mode, all rows otherwise
                const int64_t mrow = a.scratch_parts != nullptr ? i : a.row_offset + i;
                if (a.gk != nullptr) g += a.gk[i] * a.mu_all[mrow * a.ldmu + dd];
                if (a.eps != nullptr) g += gz;
                const int64_t grow = a.scratch_parts != nullptr ? i : a.row_offset + i;     // grad_mu covers the local rows only in the peer mode
                a.grad_mu[grow * a.ldgmu + dd] = g;
            }
        } else {
            const int64_t k = idx - n_row;
            const int j = (int)(k / a.d), dd = (int)(k % a.d);
            const int i = j - a.row_offset;
            const bool local = i >= 0 && i < a.b_loc;
            if (local && rows_own_mu) continue;
            float g = -kTwoLn2 * a.Gpart[(size_t)j * a.dp + dd];
            if (a.gk != nullptr && local) g += a.gk[i] * a.mu_all[(int64_t)j * a.ldmu + dd];
            a.grad_mu[(int64_t)j * a.ldgmu + dd] = g;
        }
    }
}

__device__ __forceinline__ float4 ld_volatile_f4(const void* p) {                 // peer-mapped memory: no L1 / nc path
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }

// The same finalize with 16-byte accesses (4 dims per thread): launched when d % 4 == 0 and every caller-side pitch / pointer is
// 16-byte aligned; bwd_fused_finalize_kernel covers the rest.  At one rank of eight the step spends as long in its small kernels
// as in 5 % of its sweeps, so their memory-level parallelism matters there.
__global__ void bwd_fused_finalize_v4_kernel(const BwdFinArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int d4 = a.d / 4;
    const int64_t n_row = (int64_t)a.b_loc * d4;
    const int64_t n_col = a.scratch_parts != nullptr ? 0 : (int64_t)a.b_glob * d4;
    const size_t split_stride = (size_t)a.bl_pad * a.dp;
    const bool rows_own_mu = a.scratch_parts != nullptr || a.eps != nullptr;
    if (a.scratch_parts != nullptr && a.sync.on()) peer_barrier(a.sync);
    auto ld4 = [](const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); };
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_row + n_col; idx += (int64_t)gridDim.x * blockDim.x) {
        if (idx < n_row) {
            const int i = (int)(idx / d4), dd = 4 * (int)(idx % d4);
            const size_t o = (size_t)i * a.dp + dd;
            float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sc = sa;
            const int64_t qb = (int64_t)(dd / a.slice_dp) * a.n_rb + i / a.rows_per_block;
            const int n_slots = seg_slots(a.seg, qb, a.tiles_per_block);
            for (int s0 = 0; s0 < n_slots; s0 += 4) {
                float4 va[4], vc[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool ok = s0 + k < n_slots;
                    va[k] = ok ? ld4(a.Apart + (size_t)(s0 + k) * split_stride + o) : make_float4(0.f, 0.f, 0.f, 0.f);
                    vc[k] = ok ? ld4(a.CRpart + (size_t)(s0 + k) * split_stride + o) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) { sa = f4_add(sa, va[k]); sc = f4_add(sc, vc[k]); }
            }
            const float4 vr = ld4(a.vr + o), ns = ld4(a.ns + o);
            float glv[4] = {vr.x * (kTwoLn2 * sc.x), vr.y * (kTwoLn2 * sc.y), vr.z * (kTwoLn2 * sc.z), vr.w * (kTwoLn2 * sc.w)};
            const float gz[4] = {kTwoLn2 * ns.x * sa.x, kTwoLn2 * ns.y * sa.y, kTwoLn2 * ns.z * sa.z, kTwoLn2 * ns.w * sa.w};
            float lv[4] = {0.f, 0.f, 0.f, 0.f};
            if (a.gk != nullptr || a.eps != nullptr) {
                const float4 l4 = *reinterpret_cast<const float4*>(a.lv + (int64_t)i * a.ldlv + dd);
                lv[0] = l4.x; lv[1] = l4.y; lv[2] = l4.z; lv[3] = l4.w;
            }
            if (a.gk != nullptr) {
                const float gk = a.gk[i];
#pragma unroll
                for (int e = 0; e < 4; ++e) glv[e] += gk * 0.5f * (expf(lv[e]) - 1.0f);
            }
            if (a.eps != nullptr) {                                                  // through z = mu + eps*std
                const float4 e4 = *reinterpret_cast<const float4*>(a.eps + (int64_t)i * a.ldeps + dd);
                const float ev[4] = {e4.x, e4.y, e4.z, e4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) glv[e] += gz[e] * ev[e] * (0.5f * expf(0.5f * lv[e]));
            }
            *reinterpret_cast<float4*>(a.grad_z + (int64_t)i * a.ldgz + dd) = make_float4(gz[0], gz[1], gz[2], gz[3]);
            *reinterpret_cast<float4*>(a.grad_lv + (int64_t)i * a.ldglv + dd) = make_float4(glv[0], glv[1], glv[2], glv[3]);
            if (rows_own_mu) {
                const size_t og = (size_t)(a.row_offset + i) * a.dp + dd;
                float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
                if (a.scratch_parts != nullptr) {
                    // reduce-scatter of the column gradient as this kernel's load phase: 16-byte loads of the local rows of every rank's accumulator
                    for (int p0 = 0; p0 < a.n_ranks; p0 += 8) {
                        float4 v[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            v[k] = (p0 + k < a.n_ranks) ? ld_volatile_f4(static_cast<const char*>(a.scratch_parts[p0 + k]) + a.g_off + og * sizeof(float))
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                        for (int k = 0; k < 8; ++k) g = f4_add(g, v[k]);
                    }
                } else {
                    g = ld4(a.Gpart + og);
                }
                g = f4_scale(g, -kTwoLn2);
                const int64_t mrow = a.scratch_parts != nullptr ? i : a.row_offset + i;      // mu_all = this rank's rows only in the peer mode
                if (a.gk != nullptr) g = f4_add(g, f4_scale(*reinterpret_cast<const float4*>(a.mu_all + mrow * a.ldmu + dd), a.gk[i]));
                if (a.eps != nullptr) g = f4_add(g, make_float4(gz[0], gz[1], gz[2], gz[3]));
                *reinterpret_cast<float4*>(a.grad_mu + mrow * a.ldgmu + dd) = g;              // grad_mu covers the local rows only in the peer mode
            }
        } else {
            const int64_t k = idx - n_row;
            const int j = (int)(k / d4), dd = 4 * (int)(k % d4);
            const int i = j - a.row_offset;
            const bool local = i >= 0 && i < a.b_loc;
            if (local && rows_own_mu) continue;
            float4 g = f4_scale(ld4(a.Gpart + (size_t)j * a.dp + dd), -kTwoLn2);
            if (a.gk != nullptr && local) g = f4_add(g, f4_scale(*reinterpret_cast<const float4*>(a.mu_all + (int64_t)j * a.ldmu + dd), a.gk[i]));
            *reinterpret_cast<float4*>(a.grad_mu + (int64_t)j * a.ldgmu + dd) = g;
        }
    }
}

cudaError_t launch_bwd_fused(const Plan& p, const BwdFusedArgs& a, cudaStream_t st) {
    switch (p.bwd_cfg) {
        case 0: return launch_bwd_ds_t<0>(p, a, st);
        case 1: return launch_bwd_ds_t<1>(p, a, st);
        case 2: return launch_bwd_ds_t<2>(p, a, st);
        case 3: return launch_bwd_ds_t<3>(p, a, st);
        case 4: return launch_bwd_ds_t<4>(p, a, st);
        case 5: return launch_bwd_ds_t<5>(p, a, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_bwd_fused_finalize(const Plan& p, const BwdFinArgs& a, cudaStream_t st) {
    auto ok16 = [](const void* ptr, int64_t ld) { return ptr == nullptr || ((reinterpret_cast<uintptr_t>(ptr) & 15u) == 0 && ld % 4 == 0); };
    const bool vec = p.d % 4 == 0 && ok16(a.grad_z, a.ldgz) && ok16(a.grad_lv, a.ldglv) && ok16(a.grad_mu, a.ldgmu) && ok16(a.mu_all, a.ldmu)
                     && ok16(a.lv, a.ldlv) && ok16(a.eps, a.ldeps) && (a.g_off % 16 == 0);
    const int64_t n = ((int64_t)p.b_loc * p.d + (int64_t)p.b_glob * p.d) / (vec ? 4 : 1);
    int64_t g = (n + 255) / 256; if (g > 148 * 16) g = 148 * 16; if (g < 1) g = 1;
    LaunchScope scope(kKernNone, st);
    return launch_pdl(vec ? bwd_fused_finalize_v4_kernel : bwd_fused_finalize_kernel, dim3((int)g), dim3(256), 0, st, a);
}

}  // namespace tcelbo
