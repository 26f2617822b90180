// Tensor memory (Blackwell, 256 KB per SM, otherwise idle in this library: there is no MMA anywhere) as per-thread
// scratch.  A warp may read and write the 32 TMEM lanes of its quarter (warp index % 4) with tcgen05.ld / tcgen05.st in
// the 32x32b shape: thread i of the warp owns lane 32 * (warp % 4) + i, and one instruction moves N consecutive 32-bit
// columns of that lane to / from N registers.  dls_spec.cuh parks the configuration registers of a problem there while
// the solve phases run (the compiler otherwise spills them to local memory, which an SM whose L1 is all shared memory
// serves from L2): one x32 instruction per direction instead of 14 LDL / STL pairs, and no HBM-side traffic at all.
// Device only (sm_100a); the instructions are .sync.aligned: every call must be reached by all 32 lanes of the warp.
#pragma once
#include <cstdint>

namespace ikb {

// One warp of the CTA allocates `cols` columns (a power of two >= 32) and publishes the base address at `slot` (shared
// memory); everybody reads it after the barrier.  Returns the base address.
template <int COLS> __device__ __forceinline__ uint32_t tmem_provision(uint32_t *slot, int warp) {
    static_assert(COLS == 32 || COLS == 64 || COLS == 128 || COLS == 256 || COLS == 512, "TMEM allocations are powers of two >= 32 columns");
    if (warp == 0) {
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(slot);
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"((uint32_t)COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t base = *reinterpret_cast<volatile uint32_t *>(slot);
    __syncthreads();  // the slot may be reused
    return base;
}
template <int COLS> __device__ __forceinline__ void tmem_release(uint32_t base, int warp) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();  // nobody touches tensor memory any more
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"((uint32_t)COLS) : "memory");
}

// 32 columns of the calling thread's lane <-> 32 registers
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(addr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t addr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
        "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        :
        : "r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
          "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]),
          "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// N <= 16 doubles of a thread <-> its 32 columns
template <int N> __device__ __forceinline__ void tmem_park(uint32_t addr, const double (&v)[N]) {
    static_assert(N <= 16, "one x32 transfer carries 16 doubles");
    uint32_t r[32];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        r[2 * i] = i < N ? (uint32_t)__double2loint(v[i < N ? i : 0]) : 0u;
        r[2 * i + 1] = i < N ? (uint32_t)__double2hiint(v[i < N ? i : 0]) : 0u;
    }
    tmem_st32(addr, r);
}
template <int N> __device__ __forceinline__ void tmem_fetch(uint32_t addr, double (&v)[N]) {
    static_assert(N <= 16, "one x32 transfer carries 16 doubles");
    uint32_t r[32];
    tmem_ld32(addr, r);
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __hiloint2double((int)r[2 * i + 1], (int)r[2 * i]);
}
// A thread-private strip in tensor memory with the interface of Strip (spec_common.hpp): element k of the calling thread
// lives in columns [base + k * kStride, + kStride) of its lane.  The generated bodies use it for the rows of the task
// Jacobian a warp role evaluates, factorises against and steps with -- data no other warp ever reads -- which frees
// that much shared memory for a second group of problems per SM (humanoid: 303 of 706 doubles per problem).
// set() is asynchronous (flush() before the first get of what was written); get() waits for its own load.
template <typename T> struct TStrip {
    static_assert(sizeof(T) == 8, "tensor-memory strips hold doubles (two 32-bit columns per element)");
    static constexpr int kStride = 2;
    uint32_t base;
    __device__ __forceinline__ void set(int k, T v) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(base + (uint32_t)(k * 2)), "r"((uint32_t)__double2loint(v)),
                     "r"((uint32_t)__double2hiint(v))
                     : "memory");
    }
    __device__ __forceinline__ T get(int k) const {
        uint32_t lo, hi;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(base + (uint32_t)(k * 2)) : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        return __hiloint2double((int)hi, (int)lo);
    }
    // elements k .. k + N - 1 with ONE wait: power-of-two runs of columns per tcgen05.ld, then tcgen05.wait::ld (a block
    // of generated code that reads several consecutive slots pays one tensor-memory latency instead of N)
    template <int N> __device__ __forceinline__ void getn(int k, T (&v)[N]) const {
        uint32_t r[2 * N];
        tmem_ld_run<2 * N>(base + (uint32_t)(k * 2), r);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 2 * N; ++i) asm volatile("" : "+r"(r[i]));   // no use of a loaded register moves above the wait
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = __hiloint2double((int)r[2 * i + 1], (int)r[2 * i]);
    }
    __device__ __forceinline__ void flush() const { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

  private:
    template <int C> __device__ __forceinline__ static void ld_cols(uint32_t a, uint32_t *r) {
        if constexpr (C == 16) {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                           "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                         : "r"(a)
                         : "memory");
        } else if constexpr (C == 8) {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                         : "r"(a)
                         : "memory");
        } else if constexpr (C == 4) {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                         : "r"(a)
                         : "memory");
        } else {
            static_assert(C == 2, "runs are cut into 16, 8, 4 and 2 columns");
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
        }
    }
    template <int NC> __device__ __forceinline__ static void tmem_ld_run(uint32_t a, uint32_t *r) {
        if constexpr (NC >= 16) {
            ld_cols<16>(a, r);
            tmem_ld_run<NC - 16>(a + 16, r + 16);
        } else if constexpr (NC >= 8) {
            ld_cols<8>(a, r);
            tmem_ld_run<NC - 8>(a + 8, r + 8);
        } else if constexpr (NC >= 4) {
            ld_cols<4>(a, r);
            tmem_ld_run<NC - 4>(a + 4, r + 4);
        } else if constexpr (NC >= 2) {
            ld_cols<2>(a, r);
        }
    }
};

// (single precision has registers to spare: never parked)
template <int N> __device__ __forceinline__ void tmem_park(uint32_t, const float (&)[N]) {}
template <int N> __device__ __forceinline__ void tmem_fetch(uint32_t, float (&)[N]) {}

}  // namespace ikb
