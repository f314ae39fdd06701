// radix_sort.cu -- one-sweep LSD radix sort kernels (see radix_sort.cuh).
#include "radix_sort.cuh"

namespace dsmfm {

namespace {

constexpr uint32_t kFlagAgg = 1u << 30;    // tile's own digit count is published
constexpr uint32_t kFlagPrefix = 2u << 30; // inclusive prefix over all tiles so far is published
constexpr uint32_t kValueMask = (1u << 30) - 1;

// Lanes of the warp holding the same digit (ballot multi-split).
__device__ __forceinline__ uint32_t match_digit(uint32_t d)
{
    uint32_t peers = 0xffffffffu;
#pragma unroll
    for (int b = 0; b < kRadixBits; ++b) {
        // one predicate from a constant-mask test feeds both the ballot and the keep/flip mask
        // (written in PTX: nvcc otherwise derives the two from separate shift/and/compare chains)
        uint32_t vote, flip;
        asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
                     "and.b32 t, %2, %3;\n\t"
                     "setp.ne.u32 p, t, 0;\n\t"
                     "vote.sync.ballot.b32 %0, p, 0xffffffff;\n\t"
                     "selp.b32 %1, 0, 0xffffffff, p;\n\t}"
                     : "=r"(vote), "=r"(flip)
                     : "r"(d), "r"(1u << b));
        peers &= vote ^ flip;
    }
    return peers;
}

// All digit histograms of a sort in one pass over the keys.
__global__ void __launch_bounds__(512) radix_hist_kernel(const uint64_t *__restrict__ keys, uint64_t n, int begin_bit,
                                                         int end_bit, int npass, uint64_t *__restrict__ ghist)
{
    __shared__ uint32_t h[kMaxPasses][kRadix];
    for (int i = threadIdx.x; i < kMaxPasses * kRadix; i += blockDim.x) (&h[0][0])[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t k = keys[i];
#pragma unroll
        for (int p = 0; p < kMaxPasses; ++p) {
            if (p < npass) {
                const int shift = begin_bit + kRadixBits * p;
                const int bits = min(kRadixBits, end_bit - shift);
                const uint32_t d = (uint32_t)(k >> shift) & ((1u << bits) - 1u);
                atomicAdd(&h[p][d], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npass * kRadix; i += blockDim.x) {
        const uint32_t c = (&h[0][0])[i];
        if (c) atomicAdd((unsigned long long *)&ghist[i], (unsigned long long)c);
    }
}

// Exclusive scan of each pass's 256 counts, in place.  One CTA of 256 threads per pass.
__global__ void __launch_bounds__(kRadix) radix_scan_kernel(uint64_t *__restrict__ ghist)
{
    __shared__ uint64_t warp_sum[kRadix / 32];
    uint64_t *h = ghist + (size_t)blockIdx.x * kRadix;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t v = h[tid];
    uint64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint64_t base = 0;
    for (int w = 0; w < warp; ++w) base += warp_sum[w];
    h[tid] = base + incl - v;
}

struct SweepSmem {
    uint64_t keys[kSweepTile];                 // tile in sorted order
    uint32_t vals[kSweepTile];
    uint64_t goff[kRadix];                     // global offset of digit run minus its tile-local start
    uint16_t cnt[kSweepThreads / 32][kRadix];  // per-warp digit counters -> per-warp digit bases (<= tile size)
    uint32_t excl[kRadix];                     // tile-local start of each digit run
    uint32_t warp_sum[kRadix / 32];
    uint32_t tile;
    alignas(8) uint64_t mbar;                  // completion barrier of the bulk copy of the tile's keys
};

// ---- TMA (bulk async copy) helpers: cp.async.bulk + mbarrier, sm_90+ PTX ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t arrivals)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase)
{
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(phase)
                     : "memory");
}

// One LSD pass over one portion (<= kSweepPortion pairs) of the input.
//
// Phases of a CTA (tile of 4096 pairs): load keys -> rank inside the tile (per-warp digit counters)
// -> publish the tile's digit counts -> stage keys in sorted order in shared memory -> fetch values
// while the look-back over the preceding tiles resolves the global offsets -> stage values -> write
// both out, one contiguous burst per digit.  Key registers die before the values are fetched.
// 256 threads x 16 pairs: 64 registers, 4 CTAs = 32 warps per SM.  The kernel is bound by latency
// (shared-memory round trips of the ranking, DRAM loads), not by issue slots or bandwidth, so the warps in
// flight are what counts.  Threads 0..255 own one digit each in the scan / look-back phases.
// A whole tile's keys arrive by ONE bulk asynchronous copy (cp.async.bulk, the 1-D form of TMA) into the very
// staging buffer the sorted keys overwrite later, signalled through an mbarrier; the threads then take their keys
// from shared memory (16 conflict-free LDS.64 instead of 16 predicated LDG.64 with their address arithmetic).
// The partial last tile of a portion loads its keys from global memory.
template <bool IOTA>
__global__ void __launch_bounds__(kSweepThreads, kSweepCtasPerSm)
onesweep_kernel(const uint64_t *__restrict__ keys_in, const uint32_t *__restrict__ vals_in,
                uint64_t *__restrict__ keys_out, uint32_t *__restrict__ vals_out, uint32_t n, uint64_t iota_base,
                int shift, uint32_t mask, const uint64_t *__restrict__ base_in, uint64_t *__restrict__ base_out,
                volatile uint32_t *status, uint32_t *counter, uint32_t last_tile)
{
    constexpr int THREADS = kSweepThreads, ITEMS = kSweepItems, WARPS = THREADS / 32;
    static_assert(THREADS * ITEMS == kSweepTile && THREADS == kRadix, "one tile, one thread per digit");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SweepSmem &s = *reinterpret_cast<SweepSmem *>(smem_raw);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        s.tile = atomicAdd(counter, 1u);
        mbar_init(&s.mbar, 1);
        const uint32_t t0 = s.tile * (uint32_t)kSweepTile;
        if (n - t0 >= (uint32_t)kSweepTile) bulk_load(s.keys, keys_in + t0, kSweepTile * 8, &s.mbar); // whole tiles only
    }
    for (int i = tid; i < WARPS * kRadix / 2; i += THREADS) reinterpret_cast<uint32_t *>(&s.cnt[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = s.tile;
    const uint32_t tile_base = tile * (uint32_t)kSweepTile;
    const uint32_t valid = min((uint32_t)kSweepTile, n - tile_base);
    const uint32_t first = tile_base + warp * (32 * ITEMS) + lane;

    // warp-striped load: item k of lane l is element first + 32k, so the order
    // (warp, k, lane) is the input order and the ranking below is stable
    uint64_t key[ITEMS];
    if (valid == (uint32_t)kSweepTile) {
        mbar_wait(&s.mbar, 0);
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) key[k] = s.keys[warp * (32 * ITEMS) + 32 * k + lane];
    } else
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t idx = first + 32 * k;
        key[k] = idx < n ? keys_in[idx] : ~0ull; // padding sorts to the very end of the tile
    }

    uint16_t lpos[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t d = (uint32_t)(key[k] >> shift) & mask;
        const uint32_t peers = match_digit(d);
        const int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (lane == leader) {
            old = s.cnt[warp][d];
            s.cnt[warp][d] = (uint16_t)(old + __popc(peers));
        }
        old = __shfl_sync(0xffffffffu, old, leader);
        lpos[k] = (uint16_t)(old + __popc(peers & lanemask_lt()));
        __syncwarp();
    }
    __syncthreads();

    // thread d owns digit d: the tile's count of its digit, then -- once the scan over the digits has placed the
    // digit's run inside the tile -- the position where every warp's members of the digit start
    uint32_t total = 0, pub = 0, excl = 0;
    volatile uint32_t *mine = status + (size_t)tile * kRadix + (tid & (kRadix - 1));
    if (tid < kRadix) {
#pragma unroll
        for (int w = 0; w < WARPS; ++w) total += s.cnt[w][tid];
        // publish the tile's count of digit d as early as possible: later tiles are waiting for it
        pub = total;
        if ((uint32_t)tid == mask) pub -= (uint32_t)kSweepTile - valid; // do not publish the padding
        if (tile != 0) *mine = kFlagAgg | pub;

        uint32_t incl = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s.warp_sum[warp] = incl;
        excl = incl - total;
    }
    __syncthreads();
    if (tid < kRadix) {
        uint32_t wbase = 0;
        for (int w = 0; w < warp; ++w) wbase += s.warp_sum[w];
        excl += wbase;
        s.excl[tid] = excl;
        uint32_t run = excl; // per-warp counts -> absolute tile positions (one shared-memory read less per key below)
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const uint32_t t = s.cnt[w][tid];
            s.cnt[w][tid] = (uint16_t)run;
            run += t;
        }
    }
    __syncthreads();

    // stage the keys in sorted order; afterwards only their tile-local positions stay in registers
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t d = (uint32_t)(key[k] >> shift) & mask;
        const uint32_t p = lpos[k] + s.cnt[warp][d];
        s.keys[p] = key[k];
        lpos[k] = (uint16_t)p;
    }

    // values are fetched now so that their latency overlaps the look-back
    uint32_t val[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const uint32_t idx = first + 32 * k;
        if (IOTA)
            val[k] = (uint32_t)(iota_base + idx);
        else
            val[k] = idx < n ? vals_in[idx] : 0u;
    }

    // decoupled look-back, one chain per digit, four predecessors in flight at a time
    if (tid < kRadix) {
        uint32_t exclusive = 0;
        if (tile == 0) {
            *mine = kFlagPrefix | pub;
        } else {
            uint32_t t = tile; // next predecessor to read is t-1
            bool done = false;
            while (!done) {
                const uint32_t cnt = t < 4u ? t : 4u;
                uint32_t w[4];
#pragma unroll
                for (uint32_t j = 0; j < 4; ++j)
                    if (j < cnt) w[j] = status[(size_t)(t - 1 - j) * kRadix + tid];
#pragma unroll
                for (uint32_t j = 0; j < 4; ++j) {
                    if (j < cnt && !done) {
                        uint32_t x = w[j];
                        while ((x >> 30) == 0) x = status[(size_t)(t - 1 - j) * kRadix + tid];
                        exclusive += x & kValueMask;
                        if (x & kFlagPrefix) done = true;
                    }
                }
                t -= cnt;
            }
            *mine = kFlagPrefix | (exclusive + pub);
        }
        const uint64_t gbase = base_in[tid] + exclusive;
        s.goff[tid] = gbase - excl;
        if (tile == last_tile) base_out[tid] = gbase + pub;
    }

#pragma unroll
    for (int k = 0; k < ITEMS; ++k) s.vals[lpos[k]] = val[k];
    __syncthreads();

    // every digit run goes out as one contiguous burst
    for (uint32_t i = tid; i < valid; i += THREADS) {
        const uint64_t kk = s.keys[i];
        const uint32_t d = (uint32_t)(kk >> shift) & mask;
        const uint64_t o = s.goff[d] + i;
        keys_out[o] = kk;
        vals_out[o] = s.vals[i];
    }
}

} // namespace

void RadixWorkspace::allocate(uint64_t max_n)
{
    release();
    const uint64_t portion = max_n < kSweepPortion ? max_n : kSweepPortion;
    status_tiles = div_up(portion ? portion : 1, kSweepTile);
    DSM_CUDA(cudaMalloc(&hist, sizeof(uint64_t) * kMaxPasses * kRadix));
    DSM_CUDA(cudaMalloc(&carry, sizeof(uint64_t) * 2 * kRadix));
    DSM_CUDA(cudaMalloc(&status, sizeof(uint32_t) * status_tiles * kRadix));
    DSM_CUDA(cudaMalloc(&counter, sizeof(uint32_t)));
    bytes = sizeof(uint64_t) * (kMaxPasses + 2) * kRadix + sizeof(uint32_t) * (status_tiles * kRadix + 1);
}

void RadixWorkspace::release()
{
    if (hist) cudaFree(hist);
    if (carry) cudaFree(carry);
    if (status) cudaFree(status);
    if (counter) cudaFree(counter);
    hist = carry = nullptr;
    status = counter = nullptr;
    status_tiles = 0;
    bytes = 0;
}

int radix_sort_pairs(cudaStream_t stream, RadixWorkspace &ws, uint64_t *keys_a, uint32_t *vals_a, uint64_t *keys_b,
                     uint32_t *vals_b, uint64_t n, int begin_bit, int end_bit, bool iota_first,
                     uint32_t *launches, cudaEvent_t ev_begin, cudaEvent_t ev_end, bool hist_ready)
{
    const int npass = (int)div_up((uint64_t)(end_bit - begin_bit), kRadixBits);
    if (n == 0 || npass <= 0) return 0;
    if (npass > kMaxPasses) throw CudaError{cudaErrorInvalidValue, "radix_sort_pairs: too many passes", __FILE__, __LINE__};
    if (n >= (1ull << 32)) throw CudaError{cudaErrorInvalidValue, "radix_sort_pairs: 2^32 pairs or more", __FILE__, __LINE__};
    if (div_up(n < kSweepPortion ? n : kSweepPortion, kSweepTile) > ws.status_tiles)
        throw CudaError{cudaErrorInvalidValue, "radix_sort_pairs: workspace too small", __FILE__, __LINE__};
    if ((reinterpret_cast<uintptr_t>(keys_a) & 15) != 0 || (reinterpret_cast<uintptr_t>(keys_b) & 15) != 0)
        throw CudaError{cudaErrorInvalidValue, "radix_sort_pairs: key arrays not 16-byte aligned", __FILE__, __LINE__};

    static DeviceOnce attr_once;
    attr_once.run([] {
        for (auto kernel : {onesweep_kernel<false>, onesweep_kernel<true>}) {
            DSM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SweepSmem)));
            DSM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        }
    });

    if (!hist_ready) {
        DSM_CUDA(cudaMemsetAsync(ws.hist, 0, sizeof(uint64_t) * npass * kRadix, stream));
        uint64_t want = div_up(n, 512 * 16);
        int grid = (int)(want < (uint64_t)kNumSMs * 4 ? (want ? want : 1) : (uint64_t)kNumSMs * 4);
        radix_hist_kernel<<<grid, 512, 0, stream>>>(keys_a, n, begin_bit, end_bit, npass, ws.hist);
        DSM_LAUNCH_CHECK();
        if (launches) *launches += 1;
    }
    radix_scan_kernel<<<npass, kRadix, 0, stream>>>(ws.hist);
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 1;
    if (ev_begin) DSM_CUDA(cudaEventRecord(ev_begin, stream));
    for (int p = 0; p < npass; ++p) {
        const int shift = begin_bit + kRadixBits * p;
        const int bits = (end_bit - shift) < kRadixBits ? (end_bit - shift) : kRadixBits;
        const uint32_t mask = (1u << bits) - 1u;
        uint64_t *src_k = (p & 1) ? keys_b : keys_a, *dst_k = (p & 1) ? keys_a : keys_b;
        uint32_t *src_v = (p & 1) ? vals_b : vals_a, *dst_v = (p & 1) ? vals_a : vals_b;
        const bool iota = (p == 0 && iota_first);
        const uint64_t *base_in = ws.hist + (size_t)p * kRadix;
        int flip = 0;
        for (uint64_t start = 0; start < n; start += kSweepPortion) {
            const uint64_t cnt = (n - start) < kSweepPortion ? (n - start) : kSweepPortion;
            const uint32_t tiles = (uint32_t)div_up(cnt, kSweepTile);
            uint64_t *base_out = ws.carry + (size_t)flip * kRadix;
            DSM_CUDA(cudaMemsetAsync(ws.status, 0, sizeof(uint32_t) * (size_t)tiles * kRadix, stream));
            DSM_CUDA(cudaMemsetAsync(ws.counter, 0, sizeof(uint32_t), stream));
            // (the bulk copy of a tile's keys needs a 16-byte aligned source: portions start at multiples of 2^29 pairs)
            (iota ? onesweep_kernel<true> : onesweep_kernel<false>)<<<tiles, kSweepThreads, sizeof(SweepSmem), stream>>>(
                src_k + start, iota ? nullptr : src_v + start, dst_k, dst_v, (uint32_t)cnt, start, shift, mask, base_in,
                base_out, ws.status, ws.counter, tiles - 1);
            DSM_LAUNCH_CHECK();
            if (launches) *launches += 1;
            base_in = base_out;
            flip ^= 1;
        }
    }
    if (ev_end) DSM_CUDA(cudaEventRecord(ev_end, stream));
    return npass;
}

} // namespace dsmfm
