// Types shared by the generated topology-specialised solver bodies (ik_b200/csrc/gen/*.cuh, emitted by
// tools/gen_kernel.py) and their two consumers: the CUDA kernel in dls_spec.cuh and the g++-compiled unit-test
// harness in tests/cpu_harness (the bodies are __host__ __device__ precisely so that the same source can be checked
// against the oracle on the GPU-less build box).  Host-compilable: no CUDA headers here.
#pragma once
#include "se3_math.cuh"

// Compiler-only memory fence between the phases of the generated bodies.  The strips are there precisely to get
// values OUT of registers; without the fence nvcc forwards the shared-memory stores of one phase to the loads of the
// next (keeping ~180 doubles "in registers", i.e. spilling them to local memory).  No instruction is emitted.
#define IKB_PHASE_FENCE() asm volatile("" ::: "memory")

namespace ikb {

// Run-time constants of a specialised problem.  Passed BY VALUE as a __grid_constant__ kernel parameter, so every
// access with a compile-time index becomes a constant-bank operand of the consuming instruction (no load).
template <typename T, int NQ, int M> struct SpecConsts {
    T lower[NQ], upper[NQ];  // model.lowerPositionLimit / upperPositionLimit (common.hpp:54-55)
    T weight[M];             // Task::weighting() rows in stacked order (task.hpp:40, data.cpp:49-50)
    T mask[M];               // PostureTask::mask per row (posture.hpp:52), 1 for the rows of other tasks
};

// A thread-private strip of shared memory: element k of thread t lives at base0[k * STRIDE + t], i.e. consecutive
// lanes touch consecutive words (conflict-free for 4- and 8-byte scalars).  STRIDE = 1 gives a plain array (CPU).
template <typename T, int STRIDE> struct Strip {
    static constexpr int kStride = STRIDE;
    T *base;
    IKB_HD void set(int k, T v) const { base[k * STRIDE] = v; }
    IKB_HD T get(int k) const { return base[k * STRIDE]; }
    IKB_HD T operator[](int k) const { return base[k * STRIDE]; }
    template <int N> IKB_HD void getn(int k, T (&v)[N]) const {   // (TStrip: one tensor-memory wait for the whole run)
        for (int i = 0; i < N; ++i) v[i] = base[(k + i) * STRIDE];
    }
    IKB_HD void flush() const {}   // (TStrip, tmem_scratch.cuh: wait for the asynchronous stores)
    // element k <- *src, asynchronously on the device (cp.async: global -> shared without a register in between, so a
    // whole pose is in flight at once and its latency is paid once); the copying thread calls strip_copies_wait() before
    // it reads the strip.  The strips are only ever read by the thread that filled them, so no barrier is involved.
    IKB_HD void copy_in(int k, const T *src) const {
#if defined(__CUDA_ARCH__)
        static_assert(sizeof(T) == 4 || sizeof(T) == 8, "cp.async copies 4, 8 or 16 bytes");
        const unsigned dst = (unsigned)__cvta_generic_to_shared(base + k * STRIDE);
        if (sizeof(T) == 8)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
        else
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
#else
        base[k * STRIDE] = *src;
#endif
    }
};
IKB_HD void strip_copies_wait() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}

}  // namespace ikb
