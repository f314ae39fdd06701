// common.cuh -- shared device/host helpers for the FM-index build kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include <string>

namespace dsmfm {

// ---- error plumbing -------------------------------------------------------
struct CudaError {
    cudaError_t code;
    const char *what;
    const char *file;
    int line;
};

#define DSM_CUDA(expr)                                                          \
    do {                                                                        \
        cudaError_t _e = (expr);                                                \
        if (_e != cudaSuccess) throw ::dsmfm::CudaError{_e, #expr, __FILE__, __LINE__}; \
    } while (0)

#define DSM_LAUNCH_CHECK() DSM_CUDA(cudaGetLastError())

static inline uint64_t div_up(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// Function attributes (dynamic shared memory above 48 KB, carve-out) are per DEVICE: a process that builds on
// several GPUs (dsmfm_options.device; the multi-GPU host runs one thread per device) must set them once on each.
// run(f) calls f the first time it is reached on the current device; callers on other threads wait for it.
struct DeviceOnce {
    std::mutex mu;
    uint64_t done[4] = {0, 0, 0, 0}; // up to 256 device ordinals
    template <typename F> void run(F &&f)
    {
        int dev = 0;
        DSM_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> g(mu);
        const uint64_t bit = 1ull << (dev & 63);
        uint64_t &word = done[(dev >> 6) & 3];
        if (word & bit) return;
        f();
        word |= bit;
    }
};

// Number of SMs on B200; grids for grid-stride kernels are sized in multiples of it.
constexpr int kNumSMs = 148;

// ---- packed text ----------------------------------------------------------
// Symbols are re-coded densely (0 = terminator, 1..sigma in byte order) and
// packed BITS per symbol, most significant symbol first, SPW symbols per
// 64-bit word, so that an unsigned compare of two words is a lexicographic
// compare of SPW symbols.  BITS=3: 21 symbols in bits 62..0 (bit 63 is 0).
template <int BITS> struct Pack {
    static constexpr int SPW = 64 / BITS;                 // symbols per word: 21, 16, 8
    static constexpr int USED = SPW * BITS;               // 63, 64, 64
    static constexpr uint64_t USED_MASK = USED == 64 ? ~0ull : ((1ull << USED) - 1);
    static constexpr uint64_t FIELD = (1ull << BITS) - 1;
    // bit 0 of every field
    static constexpr uint64_t lsb_mask()
    {
        uint64_t m = 0;
        for (int i = 0; i < SPW; ++i) m |= 1ull << (i * BITS);
        return m;
    }
    static constexpr uint64_t LSB = lsb_mask();
};

// Keep the symbols of x up to and including the first terminator (a zero
// field, scanning from the most significant field) and zero everything after:
// suffix comparisons never look past a terminator (incbwt/misc/utils.cpp:362-367).
template <int BITS> __host__ __device__ __forceinline__ uint64_t cut_at_terminator(uint64_t x)
{
    using P = Pack<BITS>;
    uint64_t nz = x;
#pragma unroll
    for (int i = 1; i < BITS; ++i) nz |= x >> i;
    uint64_t z = ~nz & P::LSB; // bit 0 of each zero field
    if (z == 0) return x;
#ifdef __CUDA_ARCH__
    int q = 63 - __clzll((long long)z); // bit 0 of the most significant zero field
#else
    int q = 63 - __builtin_clzll(z);
#endif
    int top = q + BITS;
    return top >= 64 ? 0ull : (x & ~((1ull << top) - 1));
}

// True when the key's last field is zero, i.e. the key contains the terminator
// (everything after the first terminator has been zeroed).
template <int BITS> __host__ __device__ __forceinline__ bool key_terminated(uint64_t key)
{
    return (key & Pack<BITS>::FIELD) == 0;
}

// SPW-symbol window starting at symbol p of the packed text, cut at the terminator.
template <int BITS> __device__ __forceinline__ uint64_t text_window(const uint64_t *__restrict__ packed, uint64_t p)
{
    using P = Pack<BITS>;
    uint64_t w = p / P::SPW;
    int s = (int)(p - w * P::SPW);
    uint64_t x0 = __ldg(packed + w);
    uint64_t x = (x0 << (BITS * s)) & P::USED_MASK;
    if (s) {
        uint64_t x1 = __ldg(packed + w + 1);
        x |= x1 >> (BITS * (P::SPW - s));
    }
    return cut_at_terminator<BITS>(x);
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() { return (1u << (threadIdx.x & 31)) - 1; }

} // namespace dsmfm
