// Launch accounting + optional CUDA-event bracketing of one kernel class (used by bench.py's roofline leg).
#pragma once
#include <cuda_runtime.h>
#include <atomic>

namespace tcelbo {

enum KernelId { kKernNone = 0, kKernFwd = 1, kKernBwdRow = 2, kKernBwdCol = 3 };

struct Instr {
    std::atomic<long long> launches{0};
    int timed_kernel = kKernNone;          // which kernel class gets bracketed by the two events below
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
};
Instr& instr();

struct LaunchScope {                        // RAII: count the launch, record events around it when asked to
    cudaStream_t st; bool timed;
    LaunchScope(int kernel_id, cudaStream_t s) : st(s) {
        Instr& in = instr();
        in.launches.fetch_add(1, std::memory_order_relaxed);
        timed = (kernel_id != kKernNone && kernel_id == in.timed_kernel && in.ev_start && in.ev_stop);
        if (timed) cudaEventRecord(in.ev_start, st);
    }
    ~LaunchScope() { if (timed) cudaEventRecord(instr().ev_stop, st); }
};

// One cached int per CUDA device (cudaFuncSetAttribute is per device: a process that drives several GPUs must configure
// every kernel on each of them).  Races are benign: every thread computes the same value.
struct PerDevice {
    int v[64] = {};
    int& cur() { int d = 0; if (cudaGetDevice(&d) != cudaSuccess) d = 0; return v[d & 63]; }
};

// Let `kern` use `smem` bytes of dynamic shared memory (every launch of a kernel asks for the same amount), once per device.
// One instantiation, and so one cache, per kernel.
template <auto kern>
inline cudaError_t allow_dynamic_smem(size_t smem) {
    static PerDevice done_on;
    int& done = done_on.cur();
    if (done) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) done = 1;
    return e;
}

}  // namespace tcelbo
