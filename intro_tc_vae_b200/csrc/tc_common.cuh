// Shared device helpers for the TC-ELBO kernels (sm_100a only).
//
// Arithmetic conventions (DESIGN.md "Kernel arithmetic"): every log-density is handled in the base-2
// exponent domain so that one MUFU.EX2 per (i,j,d) is the only transcendental in the inner loops;
// packed f32x2 PTX (FFMA2/FMUL2/FADD2 in SASS) halves the FP32-pipe issue slots; the -50 clamp of
// ops.py:21,29 is an FMNMX on the exponent argument.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdlib>
#include <utility>

namespace tcelbo {

typedef unsigned long long u64;

constexpr float kLog2e   = 1.4426950408889634f;
constexpr float kLn2     = 0.6931471805599453f;
constexpr float kTwoLn2  = 1.3862943611198906f;
constexpr float kInvTwoLn2 = 0.72134752044448170f;     // 1 / (2 ln 2)
constexpr float kRsqrtE = 0.60653065971263342f;        // 2^(-1/(2 ln 2)) = e^(-1/2)
constexpr float kLog2Pi  = 1.8378770664093453f;   // log(2*pi)
constexpr float kVarFloor = 1e-4f;                // eps of gaussian_nll_loss at ops.py:18
constexpr float kLogpFloor = -50.0f;              // clamp at ops.py:21,29
constexpr float kK50     = 72.13475204444817f;    // 50 * log2(e)
constexpr float kNegBig  = -1.0e30f;              // "minus infinity" that keeps (m - m) finite

// ---- packed fp32x2 (Blackwell FFMA2 / FMUL2 / FADD2) -------------------------------------------------
__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r;
}
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) {
    u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}
__device__ __forceinline__ u64 fmul2(u64 a, u64 b) {
    u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d;
}
__device__ __forceinline__ u64 fadd2(u64 a, u64 b) {
    u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d;
}
// ---- MUFU / min-max ------------------------------------------------------------------------------
__device__ __forceinline__ float ex2(float x) {            // MUFU.EX2 (negation folds into the operand)
    float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
}
__device__ __forceinline__ float lg2(float x) {            // MUFU.LG2
    float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {   // NaN-propagating, like torch.clamp
    float y; asm("min.NaN.f32 %0, %1, %2;" : "=f"(y) : "f"(a), "f"(b)); return y;
}
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float y; asm("max.NaN.f32 %0, %1, %2;" : "=f"(y) : "f"(a), "f"(b)); return y;
}

// ---- un-floored Gaussian log-density of one element (ops.py:24-29), shared by the row-density kernels and the column-variance
//      finalize kernels so that their terms agree bit for bit ----------------------------------------------------------------
// lp = -0.5 * ((x - mu)^2 * exp(-lv) + lv + log 2pi), before the -50 clamp; t = x - mu and iv = exp(-lv) are returned for the
// gradient.  The roundings are spelled out so that constant operands (the prior: mu = lv = 0) cannot change them.  With
// lv < -88.7 and x == mu the product is 0 * inf = NaN, as in the reference.
__device__ __forceinline__ float lp_unfloored(float x, float mu, float lv, float& t, float& iv) {
    t = x - mu;
    iv = expf(-lv);
    return -0.5f * __fadd_rn(fmaf(__fmul_rn(t, t), iv, lv), kLog2Pi);
}
// the clamped value (max.NaN: a NaN term stays NaN, like torch.clamp) and the gradient mask of the clamp
__device__ __forceinline__ float lp_clamped(float lp) { return fmax_nan(lp, kLogpFloor); }
__device__ __forceinline__ bool lp_passes_grad(float lp) { return lp >= kLogpFloor; }

// z = mu + eps * exp(logvar / 2) (ops.py:183-185): the one formula of tcelbo_reparam_forward and of every prologue that fuses the
// reparameterize, so that a fused z has the bits of the standalone one
__device__ __forceinline__ float reparam_z(float mu, float lv, float eps) { return mu + eps * expf(0.5f * lv); }

// ---- mbarrier + 1-D bulk TMA (cp.async.bulk -> UBLKCP) -------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Wait for the phase with the given parity.  Fast path: one try_wait.  Slow path: try_wait with a suspend-time
// hint, so the hardware parks the warp until the phase completes (or ~20 us pass) instead of spinning through
// issue slots the other warps need.  Bounded: a lost transaction traps (-> CUDA error) after ~2^17 hinted waits
// (seconds) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    if (done) return;
    for (int spin = 0; ; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(addr), "r"(parity), "r"(20000u) : "memory");
        if (done) return;
        if (spin > (1 << 17)) __trap();
    }
}
// global -> shared bulk copy, completion signalled on `bar` (bytes % 16 == 0, both addresses 16B aligned)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- importance weights as ratios to the uniform weight (ops.py:42-49 without the B x B matrix) ----
struct Weights {
    float r_n;      // w(1/N) / w_uniform          (column 0)
    float r_s;      // w(strat) / w_uniform        (column 1, and column 0 of global row B-2)
    float l2r_n;    // log2 of the above
    float l2r_s;
    float lw_u;     // natural log of the uniform weight (log(1/M) for MSS, -log(B*N) for MWS)
    int   mss;      // 1: stratified weights, 0: all uniform (MWS)
    int   b_glob;
};

__device__ __forceinline__ void weight_of(const Weights& w, int i_glob, int j, float& rho, float& l2rho) {
    rho = 1.0f; l2rho = 0.0f;
    if (w.mss) {
        if (j == 0) {
            const bool odd = (i_glob == w.b_glob - 2);
            rho = odd ? w.r_s : w.r_n; l2rho = odd ? w.l2r_s : w.l2r_n;
        } else if (j == 1) {
            rho = w.r_s; l2rho = w.l2r_s;
        }
    }
    if (j >= w.b_glob) { rho = 0.0f; l2rho = -INFINITY; }
}

__device__ __forceinline__ float4 ld_volatile_v4(const float* p) {          // peer-mapped memory: no L1 / nc path
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// ---- cross-rank barrier inside a kernel, over peer-mapped flags (one process per GPU, NVLink) --------------------
// Rank r owns a flag array of n_channels * n_ranks words in memory every rank has mapped.  Barrier number e of a channel:
// every rank stores e into slot [channel][its rank] of EVERY rank's array (release, system scope) and then waits until all
// n_ranks slots of its own array have reached e (acquire).  The barrier number is `state[channel]`, a local counter that the
// PREVIOUS kernel of the stream has already advanced (the publish kernel for the forward exchange, the backward prologue
// for the backward exchange), so every CTA of the waiting kernel reads the same, stable value and no ticket is needed.
// Kernels that use this must be launched by all ranks in the same order; a rank that never arrives traps the others after
// ~30 s instead of hanging the GPUs.
struct PeerSync {
    unsigned int* const* flag_parts;   // device table [n_ranks] of the ranks' flag arrays (nullptr: no in-kernel barrier)
    unsigned int* state;               // local, zero-initialised: [channel] = number of the current barrier
    int channel, rank, n_ranks;
    __host__ __device__ __forceinline__ bool on() const { return flag_parts != nullptr; }
};

// CTA 0 signals (its first n_ranks threads), every CTA waits; call with all threads of the CTA
__device__ __forceinline__ void peer_barrier(const PeerSync& ps) {
    if ((int)threadIdx.x < ps.n_ranks) {
        const unsigned int want = *reinterpret_cast<volatile unsigned int*>(ps.state + ps.channel);
        if (blockIdx.x == 0) {
            unsigned int* dst = ps.flag_parts[threadIdx.x] + ps.channel * ps.n_ranks + ps.rank;
            asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(dst), "r"(want) : "memory");
        }
        const unsigned int* src = ps.flag_parts[ps.rank] + ps.channel * ps.n_ranks + threadIdx.x;
        const long long t0 = clock64();
        unsigned int v;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
            if ((int)(v - want) < 0 && clock64() - t0 > 60000000000ll) __trap();     // ~30 s: ranks may start seconds apart
        } while ((int)(v - want) < 0);
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel of the step starts with `pdl_trigger(); pdl_wait();`: the trigger lets the NEXT
// kernel of the stream be dispatched as soon as all CTAs of this one are running (its CTAs become resident as slots free up and
// block in their own wait), the wait returns once the PREVIOUS kernel has completed and its writes are visible.  What is saved
// is the launch latency at each of the step's kernel boundaries -- a fixed cost that matters for small shards (N = 8: 1024
// rows per GPU) and for the reference's training batch (B = 64).  Without the launch attribute both instructions are no-ops.
// TCELBO_PDL=0 launches everything fully serialised.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
    static const bool on = [] { const char* e = std::getenv("TCELBO_PDL"); return e == nullptr || std::atoi(e) != 0; }();
    return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// online logsumexp in base 2: (m, s) <- (m, s) (+) 2^x
__device__ __forceinline__ void lse2_push(float& m, float& s, float x) {
    const float mn = fmaxf(m, x);
    s = s * ex2(m - mn) + ex2(x - mn);
    m = mn;
}
__device__ __forceinline__ void lse2_merge(float& m, float& s, float m2, float s2) {
    const float mn = fmaxf(m, m2);
    s = s * ex2(m - mn) + s2 * ex2(m2 - mn);
    m = mn;
}

}  // namespace tcelbo
