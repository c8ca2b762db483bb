// TC-ELBO kernels for sm_100a: the B x B x D Gaussian log-density matrix of
// ops.py:80-84 (total_correlation -> gaussian_log_density_torch -> minibatch_stratified_sampling),
// evaluated tile by tile and reduced on the fly, forward and backward, without ever storing it.
//
// Row-variance ("active") variant, ops.py:15-21 with logvar.unsqueeze(1) (ops.py:80-82):
//   per (i,d)   s = sqrt(0.5*log2e/vc), zs = z*s, ns = -s, qmax = max(0,(50+c)*log2e), shift = max(c,-50)
//   per (i,j,d) dl = zs + ns*mu_j ; q = dl^2 ; qc = min(q,qmax) ; e = 2^-qc        (lp = shift - ln2*qc)
//   S_id = sum_j rho_ij e ; s2_ij = sum_d qc ; J2_i = log2 sum_j rho_ij 2^(-s2_ij)
// rho_ij = w_ij / w_uniform is 1 except in columns 0 and 1 (ops.py:42-49).
//
// Layout: columns (mu) are staged through shared memory by 1-D bulk TMA (cp.async.bulk + mbarrier,
// 3 stages); rows live in registers for the whole sweep.  See DESIGN.md for the thread mappings.
#include "tc_common.cuh"
#include "tc_kernels.h"
#include "tc_instr.h"

namespace tcelbo {

// =====================================================================================================
// Prologues: pad/copy the column operand, derive the per-(i,d) constants
// =====================================================================================================
// Peer exchange, forward: copy this rank's rows of mu (and, for the column-variance decomposition, of logvar: src2 -> dst2) into
// its peer-mapped buffers and open the next forward barrier (the prologue kernel that follows on the stream signals and waits on
// that number, tc_common.cuh: PeerSync).
__global__ void publish_kernel(const float* __restrict__ src, int64_t ld, const float* __restrict__ src2, int64_t ld2, int b_loc, int d,
                               float* __restrict__ dst, float* __restrict__ dst2, unsigned int* epoch) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    if (blockIdx.x == 0 && threadIdx.x == 0 && epoch != nullptr) atomicAdd(epoch, 1u);
    const int64_t n = (int64_t)b_loc * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        dst[idx] = src[(idx / d) * ld + idx % d];
        if (dst2 != nullptr) dst2[idx] = src2[(idx / d) * ld2 + idx % d];
    }
}

template <bool kParts>
__global__ void prep_scalar_kernel(const PrepArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int64_t n_col = (int64_t)a.bg_pad * a.dp, n_row = (int64_t)a.bl_pad * a.dp;
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.ticket = 0u;
    // ---- rows first (local data only): per-(i,d) constants, optionally the fused reparameterize
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_row; k += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(k / a.dp), dd = (int)(k % a.dp);
        float o_zs = 0.f, o_ns = 0.f, o_q = 0.f, o_sh = 0.f, o_vr = 0.f;
        if (i < a.b_loc && dd < a.d) {
            const float lv = a.logvar[(int64_t)i * a.ldlv + dd];
            float zv;
            if (a.eps != nullptr) {                                     // fused reparameterize, ops.py:183-185
                zv = reparam_z(a.mu_loc[(int64_t)i * a.ldmu_loc + dd], lv, a.eps[(int64_t)i * a.ldeps + dd]);
                if (a.z_out != nullptr) a.z_out[(int64_t)i * a.ldz_out + dd] = zv;
            } else {
                zv = a.z[(int64_t)i * a.ldz + dd];
            }
            const float var = expf(lv);
            const float vc = (var < kVarFloor) ? kVarFloor : var;       // NaN stays NaN, like clamp_
            const float iv = 1.0f / vc;
            const float c = -0.5f * (logf(vc) + kLog2Pi);
            const float sc = sqrtf(0.5f * kLog2e * iv);
            o_zs = zv * sc;
            o_ns = -sc;
            o_q = fmaxf(0.0f, (50.0f + c) * kLog2e);
            o_sh = (c < kLogpFloor) ? kLogpFloor : c;
            o_vr = 0.5f * var * iv;                                     // straight-through floor: d/dlv uses the unclamped var
        }
        a.zs[k] = o_zs; a.ns[k] = o_ns; a.qmax[k] = o_q; a.shift[k] = o_sh; a.vr[k] = o_vr;
    }
    // ---- columns, padded.  With kParts the rows of mu live in `rows_per_part`-row blocks of different allocations (one per rank,
    //      peer-mapped): the all-gather of the column operand is this kernel's load phase (128-byte reads over NVLink), after
    //      the in-kernel barrier that tells every rank's block is published (the row work above overlaps the wait)
    if (kParts && a.sync.on()) peer_barrier(a.sync);
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_col; idx += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(idx / a.dp), dd = (int)(idx % a.dp);
        float v = 0.0f;
        if (j < a.b_glob && dd < a.d) {
            if (kParts) {
                const int part = j / a.rows_per_part;
                v = *static_cast<const volatile float*>(a.parts[part] + (int64_t)(j - part * a.rows_per_part) * a.ld_part + dd);   // no L1 / nc path
            } else {
                v = a.mu_all[(int64_t)j * a.ldmu + dd];
            }
        }
        a.mu_pad[idx] = v;
    }
}

// The same prologue with 16-byte accesses: launched when d % 4 == 0 and every caller-side pitch / pointer is 16-byte aligned
// (the encoder's chunk views and dense tensors both are, for D % 4 == 0); prep_scalar_kernel covers the rest.
template <bool kParts>
__global__ void prep_kernel(const PrepArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int dp4 = a.dp / 4;
    const int64_t n_col = (int64_t)a.bg_pad * dp4, n_row = (int64_t)a.bl_pad * dp4;
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.ticket = 0u;
    auto ld4 = [](const float* p) { return *reinterpret_cast<const float4*>(p); };
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_row; k += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(k / dp4), dd = 4 * (int)(k % dp4);
        float o_zs[4] = {0.f, 0.f, 0.f, 0.f}, o_ns[4] = {0.f, 0.f, 0.f, 0.f}, o_q[4] = {0.f, 0.f, 0.f, 0.f}, o_sh[4] = {0.f, 0.f, 0.f, 0.f},
              o_vr[4] = {0.f, 0.f, 0.f, 0.f};
        if (i < a.b_loc && dd < a.d) {
            const float4 lv4 = ld4(a.logvar + (int64_t)i * a.ldlv + dd);
            const float lvv[4] = {lv4.x, lv4.y, lv4.z, lv4.w};
            float zv[4];
            if (a.eps != nullptr) {                                     // fused reparameterize, ops.py:183-185
                const float4 m4 = ld4(a.mu_loc + (int64_t)i * a.ldmu_loc + dd), e4 = ld4(a.eps + (int64_t)i * a.ldeps + dd);
                const float mv[4] = {m4.x, m4.y, m4.z, m4.w}, ev[4] = {e4.x, e4.y, e4.z, e4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) zv[e] = reparam_z(mv[e], lvv[e], ev[e]);
                if (a.z_out != nullptr) *reinterpret_cast<float4*>(a.z_out + (int64_t)i * a.ldz_out + dd) = make_float4(zv[0], zv[1], zv[2], zv[3]);
            } else {
                const float4 z4 = ld4(a.z + (int64_t)i * a.ldz + dd);
                zv[0] = z4.x; zv[1] = z4.y; zv[2] = z4.z; zv[3] = z4.w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float var = expf(lvv[e]);
                const float vc = (var < kVarFloor) ? kVarFloor : var;       // NaN stays NaN, like clamp_
                const float iv = 1.0f / vc;
                const float c = -0.5f * (logf(vc) + kLog2Pi);
                const float sc = sqrtf(0.5f * kLog2e * iv);
                o_zs[e] = zv[e] * sc;
                o_ns[e] = -sc;
                o_q[e] = fmaxf(0.0f, (50.0f + c) * kLog2e);
                o_sh[e] = (c < kLogpFloor) ? kLogpFloor : c;
                o_vr[e] = 0.5f * var * iv;                                  // straight-through floor: d/dlv uses the unclamped var
            }
        }
        reinterpret_cast<float4*>(a.zs)[k] = make_float4(o_zs[0], o_zs[1], o_zs[2], o_zs[3]);
        reinterpret_cast<float4*>(a.ns)[k] = make_float4(o_ns[0], o_ns[1], o_ns[2], o_ns[3]);
        reinterpret_cast<float4*>(a.qmax)[k] = make_float4(o_q[0], o_q[1], o_q[2], o_q[3]);
        reinterpret_cast<float4*>(a.shift)[k] = make_float4(o_sh[0], o_sh[1], o_sh[2], o_sh[3]);
        reinterpret_cast<float4*>(a.vr)[k] = make_float4(o_vr[0], o_vr[1], o_vr[2], o_vr[3]);
    }
    if (kParts && a.sync.on()) peer_barrier(a.sync);
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_col; idx += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(idx / dp4), dd = 4 * (int)(idx % dp4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < a.b_glob && dd < a.d) {
            if (kParts) {
                const int part = j / a.rows_per_part;
                v = ld_volatile_v4(a.parts[part] + (int64_t)(j - part * a.rows_per_part) * a.ld_part + dd);      // 16-byte loads over NVLink
            } else {
                v = ld4(a.mu_all + (int64_t)j * a.ldmu + dd);
            }
        }
        reinterpret_cast<float4*>(a.mu_pad)[idx] = v;
    }
}

// =====================================================================================================
// Forward sweep.  LPR lanes share one row (each lane owns 4*KCH of the row's dims: 16-byte chunks
// {l + LPR*k}, k = 0..KCH-1), so a warp covers 32/LPR rows and the d-sum of a pair (i,j) needs only
// log2(LPR) shuffles.  grid = (row blocks, column splits); partial results go to the workspace.
// =====================================================================================================
template <int LPR, bool kWeighted, int KCH>
__device__ __forceinline__ float fwd_one_column(const float* __restrict__ mu_row,   // smem row of column j, + 4*l
                                                 const u64 (&zs2)[2 * KCH], const u64 (&ns2)[2 * KCH], const float (&qmx)[4 * KCH],
                                                 u64 (&S2)[2 * KCH], float rho) {
    u64 acc0 = 0ull, acc1 = 0ull;
    const u64 rho2 = pack2(rho, rho);
#pragma unroll
    for (int k = 0; k < KCH; ++k) {
        const float4 m = *reinterpret_cast<const float4*>(mu_row + 4 * LPR * k);
        const u64 d01 = ffma2(pack2(m.x, m.y), ns2[2 * k], zs2[2 * k]);
        const u64 d23 = ffma2(pack2(m.z, m.w), ns2[2 * k + 1], zs2[2 * k + 1]);
        const u64 q01 = fmul2(d01, d01);
        const u64 q23 = fmul2(d23, d23);
        float q0, q1, q2, q3;
        unpack2(q01, q0, q1); unpack2(q23, q2, q3);
        q0 = fmin_nan(q0, qmx[4 * k + 0]); q1 = fmin_nan(q1, qmx[4 * k + 1]);
        q2 = fmin_nan(q2, qmx[4 * k + 2]); q3 = fmin_nan(q3, qmx[4 * k + 3]);
        u64 e01 = pack2(ex2(-q0), ex2(-q1));
        u64 e23 = pack2(ex2(-q2), ex2(-q3));
        if (kWeighted) { e01 = fmul2(e01, rho2); e23 = fmul2(e23, rho2); }
        S2[2 * k] = fadd2(S2[2 * k], e01);
        S2[2 * k + 1] = fadd2(S2[2 * k + 1], e23);
        acc0 = fadd2(acc0, pack2(q0, q1));
        acc1 = fadd2(acc1, pack2(q2, q3));
    }
    acc0 = fadd2(acc0, acc1);
    float a, b; unpack2(acc0, a, b);
    return a + b;
}

template <int LPR, bool kSpecial, int KCH>
__device__ __forceinline__ void fwd_tile(const float* __restrict__ tile, int jt, int jt0, int l, int i_glob, bool row_store,
                                         const Weights& w, const u64 (&zs2)[2 * KCH], const u64 (&ns2)[2 * KCH], const float (&qmx)[4 * KCH],
                                         u64 (&S2)[2 * KCH], float& lse_m, float& lse_s, float* __restrict__ s2_row) {
    constexpr int DP = 4 * KCH * LPR;
    constexpr int G = LPR < 4 ? LPR : 4;
    // columns per iteration: after the butterfly every lane of a row keeps ONE column's joint exponent; with 8 lanes per row and
    // 16 dims per lane (KCH == 4) 8 columns are in flight so that no two lanes keep the same one
    constexpr int NC = (LPR >= 8 && KCH == 4) ? 8 : 4;
    for (int jj = 0; jj < jt; jj += NC) {
        float part[NC];
#pragma unroll
        for (int u = 0; u < NC; ++u) {
            float rho = 1.0f, l2 = 0.0f;
            if (kSpecial) weight_of(w, i_glob, jt0 + jj + u, rho, l2);
            part[u] = fwd_one_column<LPR, kSpecial, KCH>(tile + (jj + u) * DP + 4 * l, zs2, ns2, qmx, S2, rho);
        }
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) {
#pragma unroll
            for (int u = 0; u < NC; ++u) part[u] += __shfl_xor_sync(0xffffffffu, part[u], o);
        }
        if (LPR >= 4) {
            const int u = l & (NC - 1);
            float mine = part[0];
#pragma unroll
            for (int v = 1; v < NC; ++v) mine = (u == v) ? part[v] : mine;
            const int j = jt0 + jj + u;
            float x = -mine;
            if (kSpecial) { float rho, l2; weight_of(w, i_glob, j, rho, l2); x += l2; }
            lse2_push(lse_m, lse_s, x);
            if (s2_row != nullptr && row_store && l < NC) s2_row[j] = mine;
        } else {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if ((u & (G - 1)) == (l & (G - 1))) {
                    const int j = jt0 + jj + u;
                    float x = -part[u];
                    if (kSpecial) { float rho, l2; weight_of(w, i_glob, j, rho, l2); x += l2; }
                    lse2_push(lse_m, lse_s, x);
                    if (s2_row != nullptr && row_store) s2_row[j] = part[u];
                }
            }
        }
    }
}

// JTS: columns per tile (0 = as many as fit kTileFloats, at most 32); KCH: 16-byte chunks (4 dims) per lane -- 4 in the shipped
// mapping (16 dims per lane, 128 registers, 16 warps per SM), 8 (32 dims per lane, 168 registers, 3 CTAs of 4 warps per SM) in the
// small-problem instantiation; MINB: CTAs per SM; NWF: warps per CTA (8 for D >= 256, so that a CTA keeps 16 / 8 rows)
template <int LPR, int JTS, int KCH = 8, int MINB = 3, int NWF = kFwdWarps>
__global__ void __launch_bounds__(NWF * 32, MINB)
tc_fwd_kernel(const FwdArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    constexpr int DP = 4 * KCH * LPR;
    constexpr int RPW = 32 / LPR;
    constexpr int ROWS = NWF * RPW;
    constexpr int JT = JTS > 0 ? JTS : ((kTileFloats / DP) > 32 ? 32 : (kTileFloats / DP));
    constexpr int TILE = JT * DP;
    constexpr int G = LPR < 4 ? LPR : 4;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tiles = reinterpret_cast<float*>(smem_raw);                       // [kStages][TILE]
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * TILE * sizeof(float));
    uint64_t* bar_empty = bar_full + kStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int l = lane % LPR, rw = lane / LPR;
    // Work = row blocks x T column tiles, linearised block-major and cut into equal contiguous segments of a.seg.base
    // (+1) tiles, one per CTA (tc_layout.h: plan_segments): every CTA carries the same load whatever the batch shape.  A
    // segment that crosses into the next row block flushes its partial sums and reloads the row constants.
    const int T = a.bg_pad / JT;
    const int64_t g_begin = seg_begin(a.seg, blockIdx.x);
    const int ntiles = seg_len(a.seg, blockIdx.x);
    int rb = (int)(g_begin / T);
    int t_in = (int)(g_begin - (int64_t)rb * T);                             // column tile inside the current row block
    int row = rb * ROWS + warp * RPW + rw;                                   // < bl_pad by construction
    const bool row_valid = true;   // padded rows hold finite zeros: store their s2 too so backward never reads garbage

    u64 zs2[2 * KCH], ns2[2 * KCH], S2[2 * KCH];
    float qmx[4 * KCH];
    float lse_m = kNegBig, lse_s = 0.0f;
    // ---- this thread's slice of the row constants -> registers
    auto load_row = [&]() {
        const float* pz = a.zs + (size_t)row * DP + 4 * l;
        const float* pn = a.ns + (size_t)row * DP + 4 * l;
        const float* pq = a.qmax + (size_t)row * DP + 4 * l;
#pragma unroll
        for (int k = 0; k < KCH; ++k) {
            const float4 vz = __ldg(reinterpret_cast<const float4*>(pz + 4 * LPR * k));
            const float4 vn = __ldg(reinterpret_cast<const float4*>(pn + 4 * LPR * k));
            const float4 vq = __ldg(reinterpret_cast<const float4*>(pq + 4 * LPR * k));
            zs2[2 * k] = pack2(vz.x, vz.y); zs2[2 * k + 1] = pack2(vz.z, vz.w);
            ns2[2 * k] = pack2(vn.x, vn.y); ns2[2 * k + 1] = pack2(vn.z, vn.w);
            qmx[4 * k] = vq.x; qmx[4 * k + 1] = vq.y; qmx[4 * k + 2] = vq.z; qmx[4 * k + 3] = vq.w;
            S2[2 * k] = 0ull; S2[2 * k + 1] = 0ull;
        }
        lse_m = kNegBig; lse_s = 0.0f;
    };
    // ---- partial results of the current row block -> slot (this CTA's ordinal among the segments that touch the block)
    auto flush_row = [&]() {
        const int slot = (int)blockIdx.x - seg_of(a.seg, (int64_t)rb * T);
        float* ps = a.Spart + ((size_t)slot * a.bl_pad + row) * DP + 4 * l;
#pragma unroll
        for (int k = 0; k < KCH; ++k) {
            float4 v;
            unpack2(S2[2 * k], v.x, v.y); unpack2(S2[2 * k + 1], v.z, v.w);
            *reinterpret_cast<float4*>(ps + 4 * LPR * k) = v;
        }
#pragma unroll
        for (int o = 1; o < ((LPR >= 8 && KCH == 4) ? 8 : G); o <<= 1) {      // lanes of a row that hold distinct partial logsumexps
            const float m2 = __shfl_xor_sync(0xffffffffu, lse_m, o);
            const float s2v = __shfl_xor_sync(0xffffffffu, lse_s, o);
            lse2_merge(lse_m, lse_s, m2, s2v);
        }
        if (l == 0) {
            float2* pj = reinterpret_cast<float2*>(a.Jpart) + (size_t)slot * a.bl_pad + row;
            *pj = make_float2(lse_m, lse_s);
        }
    };
    load_row();

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], NWF); }
        mbar_fence_init();
    }
    __syncthreads();
    if (threadIdx.x == 0 && ntiles > 0) {
        mbar_arrive_expect_tx(&bar_full[0], TILE * sizeof(float));
        bulk_g2s(tiles, a.mu_pad + (size_t)t_in * TILE, TILE * sizeof(float), &bar_full[0]);
    }

    for (int t = 0; t < ntiles; ++t, ++t_in) {
        if (t_in == T) {                                                       // segment crosses into the next row block
            flush_row();
            ++rb; t_in = 0; row += ROWS;
            load_row();
        }
        const int st = t % kStages;
        if (threadIdx.x == 0 && t + 1 < ntiles) {                              // prefetch tile t+1 (column tiles wrap at a block boundary)
            const int sn = (t + 1) % kStages;
            const int tn = (t_in + 1 == T) ? 0 : t_in + 1;
            if (t + 1 >= kStages) mbar_wait(&bar_empty[sn], (((t + 1) / kStages) - 1) & 1);
            mbar_arrive_expect_tx(&bar_full[sn], TILE * sizeof(float));
            bulk_g2s(tiles + (size_t)sn * TILE, a.mu_pad + (size_t)tn * TILE, TILE * sizeof(float), &bar_full[sn]);
        }
        mbar_wait(&bar_full[st], (t / kStages) & 1);
        const float* tile = tiles + (size_t)st * TILE;
        const int jt0 = t_in * JT;
        const bool special = (a.w.mss && jt0 == 0) || (jt0 + JT > a.w.b_glob);
        float* s2_row = (a.s2 != nullptr) ? a.s2 + (size_t)row * a.ld_s2 : nullptr;
        const int i_glob = a.row_offset + row;
        if (special) fwd_tile<LPR, true, KCH>(tile, JT, jt0, l, i_glob, row_valid, a.w, zs2, ns2, qmx, S2, lse_m, lse_s, s2_row);
        else         fwd_tile<LPR, false, KCH>(tile, JT, jt0, l, i_glob, row_valid, a.w, zs2, ns2, qmx, S2, lse_m, lse_s, s2_row);
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_empty[st]);
    }
    flush_row();
}

// One warp per row: sum the column-split partials (float4 per lane, 8 independent loads in flight), take logs,
// emit log_qz / log_qz_prod and, when asked, either the fused KL and (beta-1)*TC + KL of solvers/tc.py:83-89 (a.lv) or the
// MI / TC / dimension-wise KL decomposition of solvers/tc.py:91-144 (a.dz).  Neither mode computes the other's terms.
__global__ void fwd_finalize_kernel(const FinArgs a) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row_raw = blockIdx.x * (blockDim.x >> 5) + warp;
    const bool row_ok = row_raw < a.b_loc;
    if (!row_ok && a.red_part == nullptr) return;
    const int row = row_ok ? row_raw : a.b_loc - 1;           // surplus warps of the last CTA recompute its last row and drop the result
    float P = 0.0f, C = 0.0f;
    const size_t split_stride = (size_t)a.bl_pad * a.dp;
    int n_js = a.n_js;                                     // uniform column split, or (balanced segments) the number of
    if (a.seg.n_ctas > 0)                                  // segments that touch this row's block
        n_js = seg_slots(a.seg, row / a.rows_per_block, a.tiles_per_block);
    for (int d0 = 4 * lane; d0 < a.dp; d0 += 128) {
        const float* src = a.Spart + (size_t)row * a.dp + d0;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s0 = 0; s0 < n_js; s0 += 8) {
            float4 v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
                v[k] = (s0 + k < n_js) ? __ldg(reinterpret_cast<const float4*>(src + (size_t)(s0 + k) * split_stride))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 8; ++k) { acc.x += v[k].x; acc.y += v[k].y; acc.z += v[k].z; acc.w += v[k].w; }
        }
        if (row_ok) *reinterpret_cast<float4*>(a.S + (size_t)row * a.dp + d0) = acc;
        const float4 sh = *reinterpret_cast<const float4*>(a.shift + (size_t)row * a.dp + d0);
        const float Sv[4] = {acc.x, acc.y, acc.z, acc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (d0 + e < a.d) { P += (logf(Sv[e]) + a.lw_u) + shv[e]; C += shv[e]; }
        }
    }
    float kl = 0.0f;
    if (a.lv != nullptr) {
        for (int dd = lane; dd < a.d; dd += 32) {
            const float l = a.lv[(int64_t)row * a.ldlv + dd], m = a.mu_loc[(int64_t)row * a.ldmu + dd];
            kl += 1.0f + l - expf(l) - m * m;
        }
    }
    float condx = 0.0f, pz = 0.0f;                           // decomposition: log q(z_i|x_i) and log p(z_i), summed over d in
    if (a.dz != nullptr) {                                   // the order of rowdensity_fwd_kernel, so they equal ops.row_log_density
        const int64_t r = (int64_t)a.row_offset + row;
        for (int dd = lane; dd < a.d; dd += 32) {
            const float x = a.dz[(int64_t)row * a.lddz + dd];
            float t, iv;
            condx += lp_clamped(lp_unfloored(x, a.dmu[r * a.lddmu + dd], a.dlv[r * a.lddlv + dd], t, iv));
            pz += lp_clamped(lp_unfloored(x, 0.0f, 0.0f, t, iv));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        P += __shfl_xor_sync(0xffffffffu, P, o);
        C += __shfl_xor_sync(0xffffffffu, C, o);
        kl += __shfl_xor_sync(0xffffffffu, kl, o);
        condx += __shfl_xor_sync(0xffffffffu, condx, o);
        pz += __shfl_xor_sync(0xffffffffu, pz, o);
    }
    float red[kFinRedSlots] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};   // this row's share of the batch means
    if (lane == 0 && row_ok) {
        const float2* pj = reinterpret_cast<const float2*>(a.Jpart);
        float m = kNegBig, s = 0.0f;
        for (int k = 0; k < n_js; ++k) {
            const float2 v = pj[(size_t)k * a.bl_pad + row];
            const float mn = fmaxf(m, v.x);
            s = s * exp2f(m - mn) + v.y * exp2f(v.x - mn);
            m = mn;
        }
        const float J2 = m + log2f(s);
        const float lq = kLn2 * J2 + C + a.lw_u;
        a.J2[row] = J2;
        if (a.log_qz != nullptr) a.log_qz[row] = lq;
        if (a.log_qz_prod != nullptr) a.log_qz_prod[row] = P;
        if (a.lv != nullptr) {                               // red = (loss, kl, -, -, exp-ELBO)
            kl *= -0.5f;
            a.kl_rows[row] = kl;
            const float loss_i = (a.beta - 1.0f) * (lq - P) + kl;
            red[0] = loss_i; red[1] = kl;
            a.loss_rows[row] = loss_i;
        } else if (a.dz != nullptr) {                        // red = (loss, mi, tc, dimkl, exp-ELBO)
            const float mi = condx - lq, tc = lq - P, dimkl = P - pz;
            red[0] = mi + a.beta * tc + dimkl; red[1] = mi; red[2] = tc; red[3] = dimkl;
            a.dec_loss[row] = red[0]; a.dec_mi[row] = mi; a.dec_tc[row] = tc; a.dec_dimkl[row] = dimkl;
        }
        if (a.rec_rows != nullptr) {                         // soft-intro exp-ELBO term of either loss (red[0] = loss_i)
            red[4] = expf(-2.0f * a.scale * (a.rec_rows[row] + red[0]));
            a.e_rows[row] = red[4];
        }
    }
    if (a.red_part == nullptr) return;
    // ---- batch means: per-CTA partials in a fixed slot, summed in fixed order by the last CTA to arrive (deterministic)
    __shared__ float sh[kFinRedSlots][kFinWarps];
    __shared__ bool last;
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < kFinRedSlots; ++q) sh[q][warp] = red[q];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < kFinRedSlots; ++q) {
            float tq = 0.0f;
            for (int w = 0; w < kFinWarps; ++w) tq += sh[q][w];
            a.red_part[q * gridDim.x + blockIdx.x] = tq;
        }
        __threadfence();
        last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!last || warp != 0) return;
    __threadfence();
    float t[kFinRedSlots] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    for (int k = lane; k < (int)gridDim.x; k += 32) {
#pragma unroll
        for (int q = 0; q < kFinRedSlots; ++q) t[q] += *(volatile float*)(a.red_part + q * gridDim.x + k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int q = 0; q < kFinRedSlots; ++q) t[q] += __shfl_xor_sync(0xffffffffu, t[q], o);
    }
    if (lane == 0) {
        const float inv_b = 1.0f / (float)a.b_loc;
        if (a.loss_mean) a.loss_mean[0] = t[0] * inv_b;
        if (a.kl_mean) a.kl_mean[0] = t[1] * inv_b;
        if (a.expelbo) a.expelbo[0] = t[4] * inv_b;
        if (a.dec_means) {
#pragma unroll
            for (int q = 0; q < 4; ++q) a.dec_means[q] = t[q] * inv_b;
        }
        *a.ticket = 0u;
    }
}

// =====================================================================================================
// Backward.  r_ijd = (gJ_i q_ij + gP_i p_ijd) m_ijd with p = rho e / S, q_ij = rho 2^(-s2_ij - J2_i),
// m = [q <= qmax] (gradient mask of the -50 clamp).  Two sweeps recompute e:
//   row pass   (rows in registers, columns streamed): A_id = sum_j r dl,  CR_id = sum_j r (2 ln2 q - 1)
//   column pass(columns in registers, rows streamed): G_jd = sum_i r dl ns_id
// Thread mapping for both: the 32 lanes of a warp span the latent dims (VEC consecutive dims per lane
// and chunk), so accumulators never cross lanes and no shuffles are needed.
// =====================================================================================================
__global__ void bwd_prep_kernel(const BwdUpstream u, const float* __restrict__ S, int b_loc, int bl_pad, int dp,
                                float* __restrict__ gps, float* __restrict__ gj, float* __restrict__ gk,
                                float* __restrict__ zero, int64_t zero_n) {
    pdl_trigger(); pdl_wait();                               // programmatic dependent launch, tc_common.cuh
    const int64_t n = (int64_t)bl_pad * dp;
    const float inv_b = 1.0f / (float)b_loc;
    const float gl_mean = u.g_loss_mean ? u.g_loss_mean[0] * inv_b : 0.0f;
    const float gk_mean = u.g_kl_mean ? u.g_kl_mean[0] * inv_b : 0.0f;
    const float ge = u.g_expelbo ? u.g_expelbo[0] * (-2.0f * u.scale * inv_b) : 0.0f;
    const float gm_mean = u.g_dec_means ? u.g_dec_means[0] * inv_b : 0.0f;      // decomposition: d/d of the mi, tc, dimkl means
    const float gt_mean = u.g_dec_means ? u.g_dec_means[1] * inv_b : 0.0f;
    const float gd_mean = u.g_dec_means ? u.g_dec_means[2] * inv_b : 0.0f;
    auto g_term = [](const float* rows, float mean, int i) { return (rows ? rows[i] : 0.0f) + mean; };
    if (u.epoch != nullptr && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(u.epoch, 1u);   // opens the backward exchange's barrier
    auto g_loss_of = [&](int i, float& g_rec) {                 // dLoss/dloss_rows[i]; g_rec = its exp-ELBO part (= dLoss/drec_rows[i])
        g_rec = u.g_expelbo ? ge * u.e_rows[i] : 0.0f;
        return (u.g_loss ? u.g_loss[i] : 0.0f) + gl_mean + g_rec;
    };
    // all arrays here are the library's own ([rows][dp] with dp % 32 == 0, 256-byte aligned): 16-byte accesses throughout
    const int64_t n4 = n / 4, zero4 = zero_n / 4, total4 = n4 > zero4 ? n4 : zero4;
    const int dp4 = dp / 4;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total4; idx += (int64_t)gridDim.x * blockDim.x) {
        if (idx < zero4) reinterpret_cast<float4*>(zero)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (idx >= n4) continue;
        const int i = (int)(idx / dp4);
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < b_loc) {
            float g_rec, gP = 0.0f;
            if (u.g_log_qz_prod) gP += u.g_log_qz_prod[i];
            gP -= (u.beta - 1.0f) * g_loss_of(i, g_rec);
            if (u.gpz) gP += g_term(u.g_dimkl, gd_mean, i) - g_term(u.g_tc, gt_mean, i);
            const float4 sv = reinterpret_cast<const float4*>(S)[idx];
            o = make_float4(gP / sv.x, gP / sv.y, gP / sv.z, gP / sv.w);
        }
        reinterpret_cast<float4*>(gps)[idx] = o;
    }
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < bl_pad; idx += (int64_t)gridDim.x * blockDim.x) {
        float gJ = 0.0f, k = 0.0f;
        if (idx < b_loc) {
            float g_rec;
            const float gl = g_loss_of((int)idx, g_rec);
            if (u.g_log_qz) gJ += u.g_log_qz[idx];
            gJ += (u.beta - 1.0f) * gl;
            k = gl + gk_mean;
            if (u.g_kl) k += u.g_kl[idx];
            if (u.g_rec_rows) u.g_rec_rows[idx] = g_rec;
            if (u.gpz) {                                                  // k is gc, the coefficient of condx
                const float gm = g_term(u.g_mi, gm_mean, (int)idx), gd = g_term(u.g_dimkl, gd_mean, (int)idx);
                gJ += g_term(u.g_tc, gt_mean, (int)idx) - gm;
                k = gl + gm;
                u.gpz[idx] = -(gl + gd);
            }
        }
        gj[idx] = gJ;
        if (gk) gk[idx] = k;
    }
}

// =====================================================================================================
// Launchers
// =====================================================================================================
static inline int grid_for(int64_t n, int block, int cap = 148 * 16) {
    int64_t g = (n + block - 1) / block;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

template <int LPR, int JTS, int KCH = 8, int MINB = 3, int NWF = kFwdWarps>
static cudaError_t launch_fwd_t(const Plan& p, const FwdArgs& a, cudaStream_t st) {
    constexpr int DP = 4 * KCH * LPR;
    constexpr int JT = JTS > 0 ? JTS : ((kTileFloats / DP) > 32 ? 32 : (kTileFloats / DP));
    constexpr auto kern = tc_fwd_kernel<LPR, JTS, KCH, MINB, NWF>;
    const size_t smem = (size_t)kStages * JT * DP * sizeof(float) + 2 * kStages * sizeof(uint64_t);
    if (cudaError_t e = allow_dynamic_smem<kern>(smem)) return e;
    LaunchScope scope(kKernFwd, st);
    return launch_pdl(kern, dim3(p.seg_fwd.n_ctas), dim3(NWF * 32), smem, st, a);
}

cudaError_t launch_publish(const float* src, int64_t ld, const float* src2, int64_t ld2, int b_loc, int d, float* dst, float* dst2,
                           unsigned int* epoch, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    return launch_pdl(publish_kernel, dim3(grid_for((int64_t)b_loc * d, 256, 148 * 4)), dim3(256), 0, st, src, ld, src2, ld2, b_loc, d,
                      dst, dst2, epoch);
}

static inline bool aligned16(const void* p, int64_t ld) { return p == nullptr || ((reinterpret_cast<uintptr_t>(p) & 15u) == 0 && ld % 4 == 0); }

cudaError_t launch_prep(const PrepArgs& a, cudaStream_t st) {
    const bool vec = a.d % 4 == 0 && aligned16(a.mu_all, a.ldmu) && aligned16(a.z, a.ldz) && aligned16(a.eps, a.ldeps)
                     && aligned16(a.mu_loc, a.ldmu_loc) && aligned16(a.z_out, a.ldz_out) && aligned16(a.logvar, a.ldlv)
                     && (a.parts == nullptr || a.ld_part % 4 == 0);          // the ranks' published buffers are dense, 16-byte aligned allocations
    LaunchScope scope(kKernNone, st);
    cudaError_t le;
    if (vec) {
        const int64_t n = (int64_t)(a.bg_pad > a.bl_pad ? a.bg_pad : a.bl_pad) * (a.dp / 4);
        if (a.parts != nullptr) le = launch_pdl(prep_kernel<true>, dim3(grid_for(n, 256)), dim3(256), 0, st, a);
        else                    le = launch_pdl(prep_kernel<false>, dim3(grid_for(n, 256)), dim3(256), 0, st, a);
    } else {
        const int64_t n = (int64_t)(a.bg_pad > a.bl_pad ? a.bg_pad : a.bl_pad) * a.dp;
        if (a.parts != nullptr) le = launch_pdl(prep_scalar_kernel<true>, dim3(grid_for(n, 256)), dim3(256), 0, st, a);
        else                    le = launch_pdl(prep_scalar_kernel<false>, dim3(grid_for(n, 256)), dim3(256), 0, st, a);
    }
    return le;
}

cudaError_t launch_fwd(const Plan& p, const FwdArgs& a, cudaStream_t st) {
    if (p.small) {
        switch (p.dpt) {
            case 1:  return launch_fwd_t<1, kSmallTile>(p, a, st);
            case 2:  return launch_fwd_t<2, kSmallTile>(p, a, st);
            case 4:  return launch_fwd_t<4, kSmallTile>(p, a, st);
            case 8:  return launch_fwd_t<8, kSmallTile>(p, a, st);
            case 16: return launch_fwd_t<16, kSmallTile>(p, a, st);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (p.fwd_lpr) {                 // 16 dims per lane, 16 warps per SM (<= 128 registers)
        case 2:  return launch_fwd_t<2, 0, 4, 4>(p, a, st);
        case 4:  return launch_fwd_t<4, 0, 4, 4>(p, a, st);
        case 8:  return launch_fwd_t<8, 0, 4, 4>(p, a, st);
        case 16: return launch_fwd_t<16, 0, 4, 2, 8>(p, a, st);      // D = 256 / 512: 8 warps per CTA keep 16 / 8 rows per CTA
        case 32: return launch_fwd_t<32, 0, 4, 2, 8>(p, a, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_fwd_finalize(const Plan& p, const FinArgs& a, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    return launch_pdl(fwd_finalize_kernel, dim3(p.n_fin_ctas), dim3(kFinWarps * 32), 0, st, a);
}

cudaError_t launch_bwd_prep(const Plan& p, const BwdUpstream& u, const float* S, float* gps, float* gj, float* gk,
                            float* zero, size_t zero_n, cudaStream_t st) {
    const int64_t n = (int64_t)p.bl_pad * p.dp;
    const int64_t total = (n > (int64_t)zero_n ? n : (int64_t)zero_n) / 4;        // one float4 per thread and pass
    LaunchScope scope(kKernNone, st);
    const cudaError_t le = launch_pdl(bwd_prep_kernel, dim3(grid_for(total, 256)), dim3(256), 0, st, u, S, p.b_loc, p.bl_pad, p.dp, gps, gj, gk, zero, (int64_t)zero_n);
    return le;
}

}  // namespace tcelbo
