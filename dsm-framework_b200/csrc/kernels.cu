// kernels.cu -- FM-index build kernels for sm_100a: ingest, key build, group
// heads, segmented refinement rounds, BWT emission, Huffman-shaped wavelet tree
// and BitRank directories.  All integer / byte work, HBM-bound; no tensor cores.
#include "kernels.cuh"
#include <cstdlib>
#include <vector>

namespace dsmfm {

namespace {

// ---------------------------------------------------------------------------
// small block-level helpers (256-thread CTAs unless noted)
// ---------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ T warp_incl_sum(T v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o) v += t;
    }
    return v;
}

template <typename T> __device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Exclusive block scan; `scratch` holds blockDim.x/32 + 1 entries; returns the
// exclusive prefix of v and puts the block total in *total.  Two barriers.
template <typename T> __device__ __forceinline__ T block_excl_sum(T v, T *scratch, T *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T incl = warp_incl_sum(v);
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    T base = 0, tot = 0;
    for (int w = 0; w < nw; ++w) {
        T s = scratch[w];
        if (w < warp) base += s;
        tot += s;
    }
    __syncthreads();
    *total = tot;
    return base + incl - v;
}

// ---------------------------------------------------------------------------
// ingest
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) byte_hist_kernel(const uint8_t *__restrict__ raw, uint64_t n,
                                                        uint64_t *__restrict__ counts)
{
    __shared__ uint32_t h[8][256];
    for (int i = threadIdx.x; i < 8 * 256; i += 256) (&h[0][0])[i] = 0;
    __syncthreads();
    uint32_t *mine = h[threadIdx.x >> 5];
    const uint64_t nvec = n / 16;
    const uint4 *v = reinterpret_cast<const uint4 *>(raw);
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < nvec; i += stride) {
        const uint4 x = __ldg(v + i);
        const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&mine[w[j] & 0xff], 1u);
            atomicAdd(&mine[(w[j] >> 8) & 0xff], 1u);
            atomicAdd(&mine[(w[j] >> 16) & 0xff], 1u);
            atomicAdd(&mine[w[j] >> 24], 1u);
        }
    }
    if (blockIdx.x == 0)
        for (uint64_t i = nvec * 16 + threadIdx.x; i < n; i += 256) atomicAdd(&mine[raw[i]], 1u);
    __syncthreads();
    uint32_t c = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) c += h[w][threadIdx.x];
    if (c) atomicAdd((unsigned long long *)&counts[threadIdx.x], (unsigned long long)c);
}

__global__ void __launch_bounds__(256) doc_stats_kernel(const uint8_t *__restrict__ raw, uint64_t n,
                                                        ChunkStat *__restrict__ out)
{
    constexpr int PER = kStatChunk / 256; // bytes per thread
    __shared__ long long s_last[8];
    __shared__ long long s_first[8];
    __shared__ unsigned long long s_max[8], s_min[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t begin = (uint64_t)blockIdx.x * kStatChunk + (uint64_t)threadIdx.x * PER;
    long long first = -1, last = -1;
    unsigned long long gmax = 0, gmin = ~0ull;
    auto terminator_at = [&](uint64_t p) {
        if (last >= 0) {
            const unsigned long long g = p - (uint64_t)last;
            gmax = g > gmax ? g : gmax;
            gmin = g < gmin ? g : gmin;
        } else {
            first = (long long)p;
        }
        last = (long long)p;
    };
    if (begin + PER <= n && (reinterpret_cast<uintptr_t>(raw) & 15) == 0) {
        // terminators are rare (one per document): test four bytes at a time
        static_assert(PER % 16 == 0, "whole 16-byte vectors per thread");
#pragma unroll
        for (int q = 0; q < PER / 16; ++q) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(raw + begin) + q);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if ((w[i] - 0x01010101u) & ~w[i] & 0x80808080u) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (((w[i] >> (8 * j)) & 0xffu) == 0) terminator_at(begin + 16 * q + 4 * i + j);
                }
            }
        }
    } else if (begin < n) {
        const uint64_t end = begin + PER < n ? begin + PER : n;
        for (uint64_t p = begin; p < end; ++p)
            if (raw[p] == 0) terminator_at(p);
    }
    // inclusive max-scan of `last` over the block -> previous terminator of each thread
    long long incl = last;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl = t > incl ? t : incl;
    }
    if (lane == 31) s_last[warp] = incl;
    __syncthreads();
    long long prev = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) prev = -1;
    for (int w = 0; w < warp; ++w) prev = s_last[w] > prev ? s_last[w] : prev;
    if (first >= 0 && prev >= 0) {
        const unsigned long long g = (uint64_t)first - (uint64_t)prev;
        gmax = g > gmax ? g : gmax;
        gmin = g < gmin ? g : gmin;
    }
    // block reductions
    long long bfirst = first >= 0 ? first : 0x7fffffffffffffffll;
    long long blast = last;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        long long f = __shfl_xor_sync(0xffffffffu, bfirst, o);
        long long l = __shfl_xor_sync(0xffffffffu, blast, o);
        unsigned long long a = __shfl_xor_sync(0xffffffffu, gmax, o);
        unsigned long long b = __shfl_xor_sync(0xffffffffu, gmin, o);
        bfirst = f < bfirst ? f : bfirst;
        blast = l > blast ? l : blast;
        gmax = a > gmax ? a : gmax;
        gmin = b < gmin ? b : gmin;
    }
    __syncthreads(); // s_last reads above are done
    if (lane == 0) {
        s_first[warp] = bfirst;
        s_last[warp] = blast;
        s_max[warp] = gmax;
        s_min[warp] = gmin;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
            bfirst = s_first[w] < bfirst ? s_first[w] : bfirst;
            blast = s_last[w] > blast ? s_last[w] : blast;
            gmax = s_max[w] > gmax ? s_max[w] : gmax;
            gmin = s_min[w] < gmin ? s_min[w] : gmin;
        }
        ChunkStat cs;
        cs.first = blast >= 0 ? bfirst : -1;
        cs.last = blast;
        cs.maxgap = gmax;
        cs.mingap = gmin;
        out[blockIdx.x] = cs;
    }
}

template <int BITS>
__global__ void __launch_bounds__(256) pack_kernel(const uint8_t *__restrict__ raw, uint64_t n,
                                                   const uint8_t *__restrict__ code_map, uint64_t *__restrict__ packed,
                                                   uint64_t nwords)
{
    using P = Pack<BITS>;
    __shared__ uint8_t map[256];
    map[threadIdx.x] = code_map[threadIdx.x];
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t w = (uint64_t)blockIdx.x * 256 + threadIdx.x; w < nwords; w += stride) {
        const uint64_t p0 = w * P::SPW;
        uint64_t x = 0;
#pragma unroll
        for (int j = 0; j < P::SPW; ++j) {
            const uint64_t p = p0 + j;
            const uint64_t c = p < n ? map[raw[p]] : 0;
            x = (x << BITS) | c;
        }
        packed[w] = x;
    }
}

// symbol code at text position q
template <int BITS> __device__ __forceinline__ uint32_t text_symbol(const uint64_t *__restrict__ packed, uint64_t q)
{
    using P = Pack<BITS>;
    const uint64_t w = q / P::SPW;
    const int s = (int)(q - w * P::SPW);
    return (uint32_t)(__ldg(packed + w) >> (BITS * (P::SPW - 1 - s))) & (uint32_t)P::FIELD;
}

// key[p] = the first `first_syms` symbols of suffix p (cut at the terminator), right-aligned in the
// low key_bits.  With carry_prev the code of the symbol BEFORE the suffix (0 at a document start) rides
// in the bits just above: the radix sort never looks at them, so the BWT symbol of every suffix
// arrives at its rank for free and no gather over the sorted suffix array is needed afterwards.
// One thread per packed word: the word and its successor hold every symbol the SPW first keys
// starting in it can need, so the keys are cut out of two registers instead of two loads and a division
// per suffix; they are staged in shared memory and leave the SM as one contiguous burst.  While the keys
// are in registers the kernel also counts their radix digits, which saves the sort's own histogram pass
// over the key array (8 bytes per suffix read back from HBM).
constexpr int kHeadsU = 8;           // head words per warp iteration of heads_kernel (8: 5.9 -> 5.3 ms on C3)
constexpr int kHeadsCtas = 4;        // resident CTAs per SM the registers of heads_kernel are budgeted for
constexpr int kKeyTileThreads = 128; // one packed word per thread and tile
constexpr int kMaxKeyPasses = 8;     // 64 key bits / 8-bit digits
constexpr int kKeySub = 1;           // copies of every digit counter in make_keys_hist_kernel (4 copies: no gain measured)

// cut_at_terminator without the early exit (same result; the keys of a whole word are cut back to back)
template <int BITS> __device__ __forceinline__ uint64_t cut_at_terminator_nb(uint64_t x)
{
    using P = Pack<BITS>;
    uint64_t nz = x;
#pragma unroll
    for (int i = 1; i < BITS; ++i) nz |= x >> i;
    const uint64_t z = ~nz & P::LSB;                 // bit 0 of each zero field
    const int top = 64 - __clzll((long long)z) + BITS - 1; // one past the most significant zero field (BITS - 1 if none)
    const uint64_t keep = z == 0 ? ~0ull : (top >= 64 ? 0ull : ~((1ull << top) - 1));
    return x & keep;
}

// Most significant bits of the fields of a 128-bit stream of BITS-bit symbols (half 0: stream bits 0..63, the first
// symbol at the top; half 1: bits 64..127).  Three-bit fields run across the two halves (the stream has its gap closed).
template <int BITS> __host__ __device__ constexpr uint64_t stream_field_msb(int half)
{
    uint64_t m = 0;
    for (int o = 0; o < 128; o += BITS)
        if (o / 64 == half) m |= 1ull << (63 - o % 64);
    return m;
}

// NP: number of 8-bit digits counted, fixed at compile time (6 for the 48-bit first key), or -1: `npass` at run time
template <int BITS, int NP>
__global__ void __launch_bounds__(kKeyTileThreads)
make_keys_hist_kernel(const uint64_t *__restrict__ packed, uint64_t n, uint64_t word_begin, uint64_t nwords,
                      uint64_t *__restrict__ keys, int key_bits, bool carry_prev, int npass_rt, uint64_t *__restrict__ ghist)
{
    using P = Pack<BITS>;
    constexpr int CAP = kKeyTileThreads * P::SPW;
    constexpr int HP = NP < 0 ? kMaxKeyPasses : (NP == 0 ? 1 : NP);
    const int npass = NP < 0 ? npass_rt : NP;
    // Read collections use few digit values (a byte of a 3-bit-per-symbol key of ACGT reads takes ~50 of its 256
    // values), so the lanes of a warp keep hitting the same counters and same-address shared atomics serialise.
    // Every counter therefore exists kKeySub times, picked by the lane: 4x fewer collisions for 18 KB more.
    constexpr int SUB = (NP > 0 && NP <= 6) ? kKeySub : 1; // (the run-time variant keeps eight tables: no room for copies)
    __shared__ uint64_t s_key[CAP];
    __shared__ uint32_t s_hist[HP][256][SUB];
    for (int i = threadIdx.x; i < HP * 256 * SUB; i += kKeyTileThreads) (&s_hist[0][0][0])[i] = 0;
    __syncthreads();
    const int sub = threadIdx.x & (SUB - 1);
    const uint64_t zkeep = key_bits >= 64 ? ~0ull : ~(~0ull >> key_bits); // the top key_bits bits
    // the words [word_begin, nwords) of the packed text (a text that streams in is keyed piece by piece)
    const uint64_t ntiles = (nwords - word_begin + kKeyTileThreads - 1) / kKeyTileThreads;
    const uint64_t n_lim = nwords * (uint64_t)P::SPW < n ? nwords * (uint64_t)P::SPW : n; // keys of later words: later calls
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint64_t w = word_begin + tile * kKeyTileThreads + threadIdx.x;
        if (w < nwords) {
            uint64_t x0 = __ldg(packed + w), x1 = __ldg(packed + w + 1); // the text is followed by zero words
            const uint32_t before = w ? (uint32_t)(__ldg(packed + w - 1) & P::FIELD) : 0u;
            if (P::USED == 63) { // 3-bit symbols sit in bits 62..0: close the gap, symbol j starts at stream bit 3j
                x0 = (x0 << 1) | (x1 >> 62);
                x1 <<= 2;
            }
            const uint64_t p0 = w * P::SPW;
            const int have = p0 + P::SPW <= n ? P::SPW : (int)(n - p0); // positions of this word inside the text
            // where the stream's fields are zero (terminators, and the zero words behind the text), once per thread:
            // a flag at the most significant bit of every zero field.  A key is cut at its first flag.
            uint64_t z0 = x0, z1 = x1;
#pragma unroll
            for (int i = 1; i < BITS; ++i) {
                z0 |= (x0 << i) | (x1 >> (64 - i));
                z1 |= x1 << i;
            }
            z0 = ~z0 & stream_field_msb<BITS>(0);
            z1 = ~z1 & stream_field_msb<BITS>(1);
#pragma unroll
            for (int j = 0; j < P::SPW; ++j) {
                if (j < have) {
                    const int b = BITS * j;
                    uint64_t v = b ? ((x0 << b) | (x1 >> (64 - b))) : x0; // stream from symbol j on
                    const uint64_t zj = (b ? ((z0 << b) | (z1 >> (64 - b))) : z0) & zkeep; // zero fields among the key's
                    if (zj) v &= ~(~0ull >> __clzll((long long)zj)); // nothing from the first terminator on
                    uint64_t k = v >> (64 - key_bits);
#pragma unroll
                    for (int q = 0; q < HP; ++q)
                        if (NP > 0 || q < npass) atomicAdd(&s_hist[q][(uint32_t)(k >> (8 * q)) & 0xffu][sub], 1u);
                    if (carry_prev) {
                        const uint32_t prev = j ? (uint32_t)((x0 >> (64 - b)) & P::FIELD) : before;
                        k |= (uint64_t)prev << key_bits;
                    }
                    s_key[threadIdx.x * P::SPW + j] = k;
                }
            }
        }
        __syncthreads();
        const uint64_t t0 = (word_begin + tile * kKeyTileThreads) * (uint64_t)P::SPW;
        const uint32_t valid = (uint32_t)(n_lim - t0 < (uint64_t)CAP ? n_lim - t0 : (uint64_t)CAP);
        for (uint32_t i = threadIdx.x; i < valid; i += kKeyTileThreads) keys[t0 + i] = s_key[i];
        __syncthreads();
    }
    for (int i = threadIdx.x; i < npass * 256; i += kKeyTileThreads) {
        uint32_t c = 0;
#pragma unroll
        for (int u = 0; u < SUB; ++u) c += (&s_hist[0][0][0])[i * SUB + u];
        if (c) atomicAdd((unsigned long long *)&ghist[i], (unsigned long long)c);
    }
}

// ---------------------------------------------------------------------------
// key-range sharding (multi-GPU): every GPU holds the whole packed text and sorts the suffixes
// whose first key falls into its range
// ---------------------------------------------------------------------------
constexpr int kSelTile = 4096; // text positions per CTA (256 threads x 16 consecutive positions)

template <int BITS>
__device__ __forceinline__ uint64_t first_key(const uint64_t *__restrict__ packed, uint64_t p, int drop_bits)
{
    return text_window<BITS>(packed, p) >> drop_bits;
}

// histogram of the top `top_bits` (<= 12) bits of the first key of every suffix
template <int BITS>
__global__ void __launch_bounds__(256)
key_top_hist_kernel(const uint64_t *__restrict__ packed, uint64_t n, int drop_bits, int top_shift,
                    unsigned long long *__restrict__ hist)
{
    __shared__ uint32_t h[4096];
    for (int i = threadIdx.x; i < 4096; i += 256) h[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x; p < n; p += stride)
        atomicAdd(&h[(uint32_t)(first_key<BITS>(packed, p, drop_bits) >> top_shift)], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < 4096; i += 256)
        if (h[i]) atomicAdd(&hist[i], (unsigned long long)h[i]);
}

// number of suffixes of each tile whose first key lies in [key_lo, key_hi)
template <int BITS>
__global__ void __launch_bounds__(256)
select_count_kernel(const uint64_t *__restrict__ packed, uint64_t n, int drop_bits, uint64_t key_lo, uint64_t key_hi,
                    uint64_t *__restrict__ tile_count)
{
    __shared__ uint32_t s_sum[8];
    const uint64_t p0 = (uint64_t)blockIdx.x * kSelTile + (uint64_t)threadIdx.x * 16;
    uint32_t c = 0;
#pragma unroll 4
    for (int j = 0; j < 16; ++j) {
        const uint64_t p = p0 + j;
        if (p < n) {
            const uint64_t k = first_key<BITS>(packed, p, drop_bits);
            c += (k >= key_lo && k < key_hi);
        }
    }
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; ++w) t += s_sum[w];
        tile_count[blockIdx.x] = t;
    }
}

// writes (key [| previous symbol above the key bits], position) of the selected suffixes in text order
template <int BITS>
__global__ void __launch_bounds__(256)
select_write_kernel(const uint64_t *__restrict__ packed, uint64_t n, int drop_bits, int key_bits, bool carry_prev,
                    uint64_t key_lo, uint64_t key_hi, const uint64_t *__restrict__ tile_off,
                    uint64_t *__restrict__ keys, uint32_t *__restrict__ vals, int lo_bits, int hi_shift)
{
    const uint64_t lo_mask = lo_bits >= 32 ? 0xffffffffull : ((1ull << lo_bits) - 1);
    __shared__ uint32_t scratch[9];
    const uint64_t p0 = (uint64_t)blockIdx.x * kSelTile + (uint64_t)threadIdx.x * 16;
    uint32_t sel = 0;
#pragma unroll 4
    for (int j = 0; j < 16; ++j) {
        const uint64_t p = p0 + j;
        if (p < n) {
            const uint64_t k = first_key<BITS>(packed, p, drop_bits);
            if (k >= key_lo && k < key_hi) sel |= 1u << j;
        }
    }
    uint32_t total;
    const uint32_t e = block_excl_sum((uint32_t)__popc(sel), scratch, &total);
    uint64_t o = tile_off[blockIdx.x] + e;
    while (sel) {
        const int j = __ffs(sel) - 1;
        sel &= sel - 1;
        const uint64_t p = p0 + j;
        uint64_t k = first_key<BITS>(packed, p, drop_bits);
        if (carry_prev && p) k |= (uint64_t)text_symbol<BITS>(packed, p - 1) << key_bits;
        // positions beyond lo_bits bits: the high part rides in the key's spare top bits (never sorted on)
        if (hi_shift) k |= (p >> lo_bits) << hi_shift;
        keys[o] = k;
        vals[o] = (uint32_t)(p & lo_mask);
        ++o;
    }
}

// ---- fast selection: one thread per packed word --------------------------------------------------
// Range membership only needs the top 12 key bits, i.e. the first kTopSyms symbols of the suffix cut at
// its terminator.  A thread takes one packed word (SPW consecutive suffixes) plus its successor as a
// 128-bit stream and classifies every suffix with a handful of 32-bit operations; the full first key
// is computed only for the suffixes that were selected.  (The generic kernels above recompute word
// index, two loads and 64-bit shifts per suffix: on G GPUs every GPU scans the whole text, so this
// scan is the part of a sharded build that does not shrink with G.)
template <int BITS> struct TopBits {
    static constexpr int SYMS = BITS == 8 ? 2 : 12 / BITS; // 4, 3, 2 symbols
    static constexpr int RAW = SYMS * BITS;                // 12, 12, 16 bits
};

// bin (top 12 key bits) of the suffix starting at symbol j of the stream s[0..3] (MSB first)
template <int BITS> __device__ __forceinline__ uint32_t top_bin(const uint32_t (&s)[4], int j)
{
    using T = TopBits<BITS>;
    const int b = BITS * j, q = b >> 5, r = b & 31;
    const uint32_t top32 = __funnelshift_l(s[q + 1 < 4 ? q + 1 : 3], s[q], r);
    uint32_t x = top32 >> (32 - T::RAW);
    // cut at the terminator: zero every field after the first zero field
    uint32_t nz = x;
#pragma unroll
    for (int i = 1; i < BITS; ++i) nz |= x >> i;
    constexpr uint32_t LSB = BITS == 3 ? 0x249u : (BITS == 4 ? 0x111u : 0x101u);
    const uint32_t z = ~nz & LSB;
    if (z) {
        const int top = 31 - __clz(z) + BITS; // bit just above the most significant zero field
        x = top >= 32 ? 0u : (x & ~((1u << top) - 1u));
    }
    return x >> (T::RAW - 12);
}

template <int BITS> __device__ __forceinline__ void load_stream(const uint64_t *__restrict__ packed, uint64_t w,
                                                                uint64_t nwords, uint32_t (&s)[4])
{
    using P = Pack<BITS>;
    uint64_t x0 = __ldg(packed + w), x1 = w + 1 < nwords ? __ldg(packed + w + 1) : 0ull;
    if (P::USED == 63) { // 3-bit symbols sit in bits 62..0: close the gap so that symbol j starts at stream bit 3j
        x0 = (x0 << 1) | (x1 >> 62);
        x1 <<= 2;
    }
    s[0] = (uint32_t)(x0 >> 32);
    s[1] = (uint32_t)x0;
    s[2] = (uint32_t)(x1 >> 32);
    s[3] = (uint32_t)x1;
}


// Selection mask of the SPW suffixes starting in a packed word: bit j set iff the bin of suffix j lies in the
// range.  The decision is read from a bitmap indexed by the RAW leading bits of the suffix (TopBits::RAW: the
// uncut first symbols), which the host fills for the range at hand -- cut at the terminator included -- so a
// suffix costs a funnel shift, a shared-memory load and a bit test instead of the whole top_bin arithmetic.
// `valid` = number of leading positions of the word that are suffixes of the collection (the rest is padding).
template <int BITS>
__device__ __forceinline__ uint32_t select_mask_lut(const uint32_t *s_lut, const uint32_t (&s)[4], int valid)
{
    using P = Pack<BITS>;
    using T = TopBits<BITS>;
    uint32_t sel = 0;
#pragma unroll
    for (int j = 0; j < P::SPW; ++j) {
        const int b = BITS * j, q = b >> 5, r = b & 31;
        const uint32_t top32 = __funnelshift_l(s[q + 1 < 4 ? q + 1 : 3], s[q], r);
        const uint32_t raw = top32 >> (32 - T::RAW);
        sel |= ((s_lut[raw >> 5] >> (raw & 31)) & 1u) << j;
    }
    return valid >= P::SPW ? sel : (sel & ((1u << valid) - 1u));
}

template <int BITS>
__global__ void __launch_bounds__(256)
key_top_hist_fast_kernel(const uint64_t *__restrict__ packed, uint64_t n, uint64_t nwords,
                         unsigned long long *__restrict__ hist)
{
    using P = Pack<BITS>;
    __shared__ uint32_t h[4096];
    for (int i = threadIdx.x; i < 4096; i += 256) h[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t w = (uint64_t)blockIdx.x * 256 + threadIdx.x; w < nwords; w += stride) {
        uint32_t s[4];
        load_stream<BITS>(packed, w, nwords, s);
        const uint64_t p0 = w * P::SPW;
        // runs of equal bins are common (a word holds consecutive suffixes of few distinct leading symbols
        // only by chance), so counts are added one by one; shared-memory atomics on 4096 bins
#pragma unroll
        for (int j = 0; j < P::SPW; ++j)
            if (p0 + j < n) atomicAdd(&h[top_bin<BITS>(s, j)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 4096; i += 256)
        if (h[i]) atomicAdd(&hist[i], (unsigned long long)h[i]);
}

// One pass: select, compute the keys of the selected suffixes and write the (key, position) pairs out in
// text order.  A CTA takes the next tile of kSweepSelWords packed words (dynamic tile id, so that a tile's
// predecessors are always running or done), counts its selected suffixes, publishes the count and obtains
// its output offset by decoupled look-back over the preceding tiles (64-bit status words: 2 flag bits + 62
// value bits); meanwhile the keys are staged in shared memory in text order, so that the tile leaves the SM
// as one contiguous burst instead of 12-byte stores scattered per thread.
constexpr int kSweepSelThreads = 128;
constexpr int kSweepSelWords = kSweepSelThreads; // one packed word per thread
constexpr unsigned long long kSelFlagAgg = 1ull << 62, kSelFlagPrefix = 2ull << 62, kSelValueMask = (1ull << 62) - 1;

// A tile is kSelSub sub-tiles of kSweepSelWords words: the selection masks of all of them are taken first (they
// stay in registers), so that the tile publishes ONE count and runs ONE look-back -- the dynamic tile id and the
// look-back are a few microseconds of latency each, which 128 words of work could not hide (the kernel spent 3.2 ms
// per G symbols on them, and on G GPUs every GPU scans the whole text) -- then the sub-tiles are staged and
// written out one after the other.
constexpr int kSelSub = 8;

template <int BITS>
__global__ void __launch_bounds__(kSweepSelThreads)
select_sweep_kernel(const uint64_t *__restrict__ packed, uint64_t nwords, int key_bits, const uint32_t *__restrict__ lut,
                    const SelGeom geom, volatile unsigned long long *status, uint32_t *counter,
                    uint64_t *__restrict__ keys, uint32_t *__restrict__ vals, int lo_bits, int hi_shift)
{
    using P = Pack<BITS>;
    using T = TopBits<BITS>;
    constexpr int CAP = kSweepSelWords * P::SPW; // suffixes per sub-tile
    constexpr int LUT_WORDS = (1 << T::RAW) / 32;
    __shared__ uint64_t s_key[CAP];
    __shared__ uint32_t s_val[CAP];
    __shared__ uint32_t s_lut[LUT_WORDS];
    __shared__ uint32_t s_w[kSelSub][kSweepSelThreads / 32];
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_base;
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid == 0) s_tile = atomicAdd(counter, 1u);
    for (int i = tid; i < LUT_WORDS; i += kSweepSelThreads) s_lut[i] = __ldg(lut + i);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t lo_mask = lo_bits >= 32 ? 0xffffffffull : ((1ull << lo_bits) - 1);
    const uint64_t w0 = (uint64_t)tile * (kSweepSelWords * kSelSub) + tid;
    // the selection masks of this thread's word in every sub-tile.  (Block and position inside the block by ONE
    // 64-bit division per thread; the other sub-tiles follow by adding the stride.)
    uint32_t sel[kSelSub];
    uint32_t mine = 0;
    uint64_t slot = w0 / geom.slot_words, rem = w0 - slot * geom.slot_words; // word rem of block `slot`
#pragma unroll
    for (int j = 0; j < kSelSub; ++j) {
        const uint64_t w = w0 + (uint64_t)j * kSweepSelWords;
        sel[j] = 0;
        if (w < nwords) {
            const uint64_t first = rem * P::SPW; // position of the word inside its block
            const uint64_t have = slot < geom.world ? geom.bytes[slot] : 0ull;
            const int valid = have > first ? (have - first >= (uint64_t)P::SPW ? P::SPW : (int)(have - first)) : 0;
            if (valid) {
                uint32_t st[4];
                load_stream<BITS>(packed, w, nwords, st);
                sel[j] = select_mask_lut<BITS>(s_lut, st, valid);
            }
        }
        mine += __popc(sel[j]);
        rem += kSweepSelWords;
        while (rem >= geom.slot_words) {
            rem -= geom.slot_words;
            ++slot;
        }
    }
    // tile-local position of this thread's first selected suffix in every sub-tile (text order: sub-tile, then thread):
    // one scan for all sub-tiles, two barriers for the whole tile
    uint32_t off[kSelSub];
#pragma unroll
    for (int j = 0; j < kSelSub; ++j) {
        const uint32_t c = __popc(sel[j]);
        const uint32_t incl = warp_incl_sum(c);
        if (lane == 31) s_w[j][tid >> 5] = incl;
        off[j] = incl - c;
    }
    __syncthreads();
    uint32_t total = 0;
#pragma unroll
    for (int j = 0; j < kSelSub; ++j) {
        uint32_t before = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kSweepSelThreads / 32; ++w) {
            const uint32_t x = s_w[j][w];
            before += w < (tid >> 5) ? x : 0u;
            tot += x;
        }
        off[j] += before + total;
        total += tot;
    }
    (void)mine;
    if (tid == 0) status[tile] = (tile == 0 ? kSelFlagPrefix : kSelFlagAgg) | total;

    // look-back by the first warp: 32 predecessors per step
    if (tid < 32) {
        unsigned long long excl = 0;
        if (tile != 0) {
            long long t = (long long)tile - 1;
            for (;;) {
                const long long idx = t - lane;
                unsigned long long x = 2ull << 62; // before the first tile: an empty prefix
                if (idx >= 0) x = status[idx];
                while (__any_sync(0xffffffffu, (x >> 62) == 0))
                    if ((x >> 62) == 0) x = status[idx];
                const uint32_t pm = __ballot_sync(0xffffffffu, (x >> 62) == 2);
                const int stop = pm ? __ffs(pm) - 1 : 32;
                unsigned long long v = lane <= stop ? (x & kSelValueMask) : 0ull;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                excl += v;
                if (pm) break;
                t -= 32;
            }
            if (lane == 0) status[tile] = kSelFlagPrefix | (excl + total);
        }
        if (lane == 0) s_base = excl;
    }
    __syncthreads();
    const uint64_t base = s_base;

    // Keys of the selected suffixes, staged in text order, CAP pairs per round (one round when an eighth of the
    // suffixes is selected, as on eight GPUs).  The word and its successor hold every symbol a first key can need
    // (first_syms <= SPW), so keys are cut out of two registers; the symbol before the suffix (the BWT symbol,
    // which rides above the key bits) is the previous symbol of the same stream.
    const uint64_t kmask = key_bits >= 64 ? ~0ull : ((1ull << key_bits) - 1);
    for (uint32_t lo = 0; lo < total; lo += CAP) {
        const uint32_t hi = lo + CAP;
#pragma unroll 1
        for (int j = 0; j < kSelSub; ++j) { // (not unrolled: eight copies of the key extraction do not fit the instruction cache)
            uint32_t sj = 0, oj = 0;
#pragma unroll
            for (int q = 0; q < kSelSub; ++q)
                if (q == j) {
                    sj = sel[q];
                    oj = off[q];
                }
            const uint32_t c = __popc(sj);
            if (c == 0 || oj >= hi || oj + c <= lo) continue;
            const uint64_t w = w0 + (uint64_t)j * kSweepSelWords;
            const uint64_t p0 = w * P::SPW;
            uint64_t x0 = __ldg(packed + w), x1 = w + 1 < nwords ? __ldg(packed + w + 1) : 0ull;
            const uint32_t before = w ? (uint32_t)(__ldg(packed + w - 1) & P::FIELD) : 0u; // last symbol of the previous word
            if (P::USED == 63) {
                x0 = (x0 << 1) | (x1 >> 62);
                x1 <<= 2;
            }
            uint32_t pos = oj;
            while (sj) {
                const int i = __ffs(sj) - 1;
                sj &= sj - 1;
                if (pos >= lo && pos < hi) {
                    const int b = BITS * i;
                    const uint64_t v = b ? ((x0 << b) | (x1 >> (64 - b))) : x0;     // stream from symbol i on
                    uint64_t k = (v >> (64 - key_bits)) | ~kmask;                  // ones above: only real fields can be zero
                    k = cut_at_terminator<BITS>(k) & kmask;
                    const uint32_t prev = i ? (uint32_t)((x0 >> (64 - b)) & P::FIELD) : before;
                    k |= (uint64_t)prev << key_bits;                               // the BWT symbol rides along
                    const uint64_t p = p0 + i;
                    if (hi_shift) k |= (p >> lo_bits) << hi_shift;
                    s_key[pos - lo] = k;
                    s_val[pos - lo] = (uint32_t)(p & lo_mask);
                }
                ++pos;
            }
        }
        __syncthreads();
        const uint32_t cnt = total - lo < (uint32_t)CAP ? total - lo : (uint32_t)CAP;
        for (uint32_t i = tid; i < cnt; i += kSweepSelThreads) {
            keys[base + lo + i] = s_key[i];
            vals[base + lo + i] = s_val[i];
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// group heads after the initial sort
// ---------------------------------------------------------------------------
// One warp per chunk of U head words (32*U consecutive ranks).  Everything a rank needs comes from its own key
// and its predecessor's (one 64-bit shuffle; the first lane of a word takes the last key of the word before):
// with x = key ^ previous key, the sorted bits of x tell whether the rank opens a group and the carried bits
// whether its BWT symbol differs.  "Next rank opens a group" is the head bit of the next rank, so the count of
// suffixes left in groups of >= 2 falls out of the head words themselves.  Chunks that lie entirely inside
// the array take a path without bounds checks and with 32-bit offsets from the chunk's base pointers.
template <int BITS>
__global__ void __launch_bounds__(256, kHeadsCtas) heads_kernel(const uint64_t *__restrict__ keys, uint64_t n,
                                                    uint32_t *__restrict__ head, uint64_t head_words,
                                                    unsigned long long *__restrict__ remaining, int key_bits,
                                                    const uint8_t *__restrict__ inv_map, uint8_t *__restrict__ bwt,
                                                    uint8_t *__restrict__ pos_hi, int hi_shift,
                                                    uint32_t *__restrict__ diff)
{
    constexpr uint64_t FIELD = Pack<BITS>::FIELD;
    constexpr int U = kHeadsU;
    __shared__ unsigned long long s_cnt[8];
    __shared__ uint8_t s_inv[256];
    if (bwt) s_inv[threadIdx.x] = inv_map[threadIdx.x];
    __syncthreads();
    const uint64_t kmask = key_bits >= 64 ? ~0ull : ((1ull << key_bits) - 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t nchunks = (head_words + U - 1) / U;
    const uint64_t warps_total = (uint64_t)gridDim.x * 8;
    // BITS = 3: the code -> byte table fits a register
    uint64_t inv_reg = 0;
    if (BITS == 3 && bwt)
        for (int c = 0; c < 8; ++c) inv_reg |= (uint64_t)s_inv[c] << (8 * c);
    uint32_t active = 0; // per lane, summed at the end (fast path) / lane 0 (slow path)
    for (uint64_t ch = (uint64_t)blockIdx.x * 8 + warp; ch < nchunks; ch += warps_total) {
        const uint64_t w0 = ch * U;
        const uint64_t base = w0 * 32; // rank of lane 0 in the chunk's first word
        if (base > 0 && base + 32 * U < n && w0 + U <= head_words) {
            // ---- all 32U ranks, the one before and the one behind exist ----
            const uint64_t *kp = keys + base;
            uint64_t k[U];
#pragma unroll
            for (int u = 0; u < U; ++u) k[u] = kp[32 * u + lane];
            uint64_t edge = 0; // lane 0: key in front of the chunk; lane 31: key behind it
            if (lane == 0) edge = kp[-1];
            if (lane == 31) edge = kp[32 * U];
            uint32_t hw[U + 1], dw[U];
            uint64_t prev_last = __shfl_sync(0xffffffffu, edge, 0);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                uint64_t kprev = __shfl_up_sync(0xffffffffu, k[u], 1);
                if (lane == 0) kprev = prev_last;
                prev_last = __shfl_sync(0xffffffffu, k[u], 31);
                const uint64_t x = k[u] ^ kprev;
                const bool h = ((x & kmask) != 0) | ((k[u] & FIELD) == 0);
                const bool df = !h & (((x >> key_bits) & FIELD) != 0);
                hw[u] = __ballot_sync(0xffffffffu, h);
                dw[u] = diff ? __ballot_sync(0xffffffffu, df) : 0u;
                if (bwt) {
                    const uint32_t code = (uint32_t)(k[u] >> key_bits) & (uint32_t)FIELD;
                    bwt[base + 32 * u + lane] = BITS == 3 ? (uint8_t)(inv_reg >> (8 * code)) : s_inv[code];
                }
                if (pos_hi) pos_hi[base + 32 * u + lane] = (uint8_t)(k[u] >> hi_shift);
            }
            {
                const uint64_t kafter = __shfl_sync(0xffffffffu, edge, 31);
                const uint64_t x = kafter ^ prev_last;
                hw[U] = (((x & kmask) != 0) | ((kafter & FIELD) == 0)) ? 1u : 0u;
            }
            // lane u stores word u; every lane counts the suffixes in groups of >= 2 of "its" word
            uint32_t myh = 0, myd = 0, mynext = 0;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (lane == u) {
                    myh = hw[u];
                    myd = dw[u];
                    mynext = (hw[u] >> 1) | (hw[u + 1] << 31);
                }
            }
            if (lane < U) {
                head[w0 + lane] = myh;
                if (diff) diff[w0 + lane] = myd;
                active += __popc(~(myh & mynext));
            }
            continue;
        }
        // ---- first chunk and the chunks around the end of the array ----
        uint64_t kraw[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t i = base + 32 * u + lane;
            kraw[u] = i < n ? keys[i] : 0ull;
        }
        const uint64_t kcarry = (base && base - 1 < n) ? keys[base - 1] : 0ull;
        const uint64_t kafter = base + 32 * U < n ? keys[base + 32 * U] : 0ull;
        uint32_t hw[U + 1];
        uint64_t prev_last = kcarry; // key of the rank in front of the current word
#pragma unroll
        for (int u = 0; u < U; ++u) {
            uint64_t kprev = __shfl_up_sync(0xffffffffu, kraw[u], 1);
            if (lane == 0) kprev = prev_last;
            prev_last = __shfl_sync(0xffffffffu, kraw[u], 31);
            const uint64_t x = kraw[u] ^ kprev;
            const uint64_t i = base + 32 * u + lane;
            bool h = (x & kmask) != 0 || key_terminated<BITS>(kraw[u] & kmask) || i == 0;
            bool df = !h && ((x >> key_bits) & FIELD) != 0;
            h = h || i >= n; // ranks behind the last suffix count as heads
            df = df && i < n;
            hw[u] = __ballot_sync(0xffffffffu, h);
            if (diff) {
                const uint32_t dw = __ballot_sync(0xffffffffu, df);
                if (lane == 0 && w0 + u < head_words) diff[w0 + u] = dw;
            }
            if (i < n) {
                if (bwt) {
                    const uint32_t code = (uint32_t)(kraw[u] >> key_bits) & (uint32_t)FIELD;
                    bwt[i] = BITS == 3 ? (uint8_t)(inv_reg >> (8 * code)) : s_inv[code];
                }
                if (pos_hi) pos_hi[i] = (uint8_t)(kraw[u] >> hi_shift); // high part of the text position (wide builds)
            }
        }
        {
            // head bit of the rank right behind the chunk
            const uint64_t i = base + 32 * U;
            const uint64_t x = kafter ^ prev_last;
            hw[U] = (i >= n || (x & kmask) != 0 || key_terminated<BITS>(kafter & kmask)) ? 1u : 0u;
        }
        if (lane == 0) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (w0 + u < head_words) {
                    head[w0 + u] = hw[u];
                    // in a group of >= 2: not (head and next rank is a head)
                    const uint32_t next = (hw[u] >> 1) | (hw[u + 1] << 31);
                    uint32_t in_group = ~(hw[u] & next);
                    const uint64_t first = (w0 + u) * 32;
                    if (first + 32 > n) in_group &= first >= n ? 0u : ((1u << (n - first)) - 1u);
                    active += __popc(in_group);
                }
            }
        }
    }
    const unsigned long long mine = warp_sum((unsigned long long)active);
    if (lane == 0) s_cnt[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 8; ++w) t += s_cnt[w];
        if (t) atomicAdd(&remaining[blockIdx.x & 63], t);
    }
}

// ---------------------------------------------------------------------------
// refinement round
// ---------------------------------------------------------------------------
// last set bit at a position <= r / first set bit at a position > r in a bit array
__device__ __forceinline__ int prev_set_le(const uint32_t *hw, int r)
{
    int w = r >> 5;
    uint32_t m = hw[w] & (0xffffffffu >> (31 - (r & 31)));
    while (m == 0) m = hw[--w];
    return (w << 5) + 31 - __clz(m);
}
__device__ __forceinline__ int next_set_gt(const uint32_t *hw, int r)
{
    int w = r >> 5;
    uint32_t m = (r & 31) == 31 ? 0u : (hw[w] & (0xffffffffu << ((r & 31) + 1)));
    while (m == 0) m = hw[++w];
    return (w << 5) + __ffs(m) - 1;
}

// SPW-symbol window that starts `s` symbols into word x0 and runs on into x1, cut at the terminator
template <int BITS> __device__ __forceinline__ uint64_t window_of(uint64_t x0, uint64_t x1, int s)
{
    using P = Pack<BITS>;
    uint64_t x = (x0 << (BITS * s)) & P::USED_MASK;
    if (s) x |= x1 >> (BITS * (P::SPW - s));
    return cut_at_terminator<BITS>(x);
}

// ---------------------------------------------------------------------------
// refinement with independent warps
// ---------------------------------------------------------------------------
// One CTA owns the groups whose head lies in its window of kRefWindow slots and keeps refining them in
// shared memory -- key = the next SPW symbols, stable rank inside the group, split -- until they are all
// resolved.  The suffix array (and the BWT bytes that travel with it) are read once; a suffix is written
// back the moment it becomes a singleton; only the text is touched again in every step.  A step is two phases:
//   rank:     every unresolved suffix finds its stable rank inside its group, moves to the other buffer
//             and marks the new group heads;
//   classify: resolved suffixes go home; the others fetch their next key and stay on the list.
// Groups never interact, so nothing forces the warps of a CTA through the steps together (CTA-wide steps
// cost two barriers each and run as many steps as the slowest suffix needs, with most warps idle in the
// tail): the CTA only shares the window in shared memory.  Warp w owns the groups whose head lies in its
// 128-slot part of the window -- a contiguous slot range [first head >= 128w, first head >= 128(w+1)) --
// and runs the rank / classify steps over that range on its own, synchronising with __syncwarp only.
// Head bits of neighbouring ranges can share a 32-bit word: words are only ever OR-ed (atomically), a
// warp publishes (head_b -> head_a) just the bits of its own range, and the bit scans stop at the
// heads that bound the range, which are set from the start.
constexpr int kRwGroupMax = kRefGroupMaxWarps;
constexpr int kRwCap = kRefWindow + kRwGroupMax;
// Groups of at least this many members are ranked by the whole warp at once.  In repetitive collections (high
// coverage, few errors) a tie group is the set of reads covering one locus: after the next 21 symbols most of
// its members still agree -- they share ONE dominant key -- and only the reads that end inside the window (or
// carry an error there) differ.  The warp counts the members below / equal to / above a candidate key with
// ballots (the equal ones get their stable rank from the running count: no comparisons among them at all) and
// ranks only the others against each other: (0.3 g)^2 comparisons instead of g^2.
constexpr int kRwBigGroup = 64;

template <bool WIDE> struct RwSmem {
    uint64_t key[kRwCap];              // the next SPW symbols of the suffix in each slot
    uint32_t sa[2][kRwCap];            // suffixes, double buffered across a step
    uint16_t list[kRwCap];             // unresolved slots of each warp's range, compacted in place
    uint8_t bw[2][kRwCap];             // BWT bytes travelling with the suffixes
    uint8_t hi[2][WIDE ? kRwCap : 1];  // wide builds: text position = hi << lo_bits | sa
    uint32_t head_a[kRwCap / 32 + 2];
    uint32_t head_b[kRwCap / 32 + 2];
    uint32_t mix[kRwCap / 32 + 2];     // per group head: the group's members carry different BWT symbols
    uint32_t df[kRwCap / 32 + 2];      // per slot: BWT symbol differs from the predecessor's inside a group
    uint32_t act[kRwCap / 32 + 2];     // per slot: member of a group that has to be sorted
    uint16_t newpos[kRwCap];           // large groups: rank of a carrier of the dominant key among the carriers
    uint16_t ghead[kRwCap];            // per slot: first slot of the group the last ranking step put its suffix in
    uint16_t nd[kRwCap];               // large groups: the members whose key is not the dominant one, in slot order
    uint16_t bigq[kRefThreads / 32][kRwCap / kRwBigGroup + 2]; // per warp: first slots of its large groups
    int range[2];
};

// ORDER = false: only the BWT is wanted, not the suffix array.  Then a tie group whose members all carry the
// same BWT symbol needs no sorting at all -- whatever their order, the BWT bytes of its slots are that symbol --
// and such groups are the rule in read collections: suffixes that agree on their next 16+ symbols mostly come
// from reads overlapping the same stretch of a genome, and they agree on the symbol in front of it too.  Only
// groups with mixed symbols are loaded and refined, and a group that becomes uniform after a split is dropped
// at once.  (ORDER = true, DSMFM_FLAG_KEEP_SA: the full order, as needed for the .sa samples.)
constexpr int kRwCtas = 4; // resident CTAs per SM the compiler budgets registers for
// COOP: groups of big_thr members or more are ranked by the whole warp around their dominant key (a separate
// instantiation: with both ranking schemes in one kernel the whole-warp path lost 10 % to the other's code).
template <int BITS, bool WIDE, bool ORDER, bool COOP>
__global__ void __launch_bounds__(kRefThreads, kRwCtas)
refine_warps_kernel(const uint64_t *__restrict__ packed, uint32_t *__restrict__ sa, const uint32_t *__restrict__ head_cur,
                    uint32_t *__restrict__ head_next, uint64_t n, uint32_t depth, const uint32_t *__restrict__ win_list,
                    uint32_t *__restrict__ big_heads, uint32_t big_cap, uint32_t *__restrict__ big_count,
                    unsigned long long *__restrict__ remaining, uint32_t *__restrict__ win_flag,
                    uint32_t *__restrict__ win_next, uint32_t *__restrict__ win_next_count, uint8_t *__restrict__ bwt,
                    uint8_t *__restrict__ sa_hi, int lo_bits, const uint32_t *__restrict__ diff_bits, int big_thr)
{
    using P = Pack<BITS>;
    constexpr int HW = kRwCap / 32 + 2;
    constexpr int WIN_WORDS = kRefWindow / 32;
    constexpr int OVER_WORDS = kRwGroupMax / 32;
    constexpr int NWARP = kRefThreads / 32;
    constexpr int PART = kRefWindow / NWARP; // slots of the window whose heads one warp owns
    static_assert(WIN_WORDS == 32 && OVER_WORDS <= 32, "one warp scans the window / the overhang");
    extern __shared__ __align__(16) unsigned char ref_smem_raw[];
    RwSmem<WIDE> &S = *reinterpret_cast<RwSmem<WIDE> *>(ref_smem_raw);
    uint64_t *s_key = S.key;
    uint32_t(*s_sa)[kRwCap] = S.sa;
    uint8_t(*s_bw)[kRwCap] = S.bw;
    uint8_t(*s_hi)[WIDE ? kRwCap : 1] = S.hi;
    uint32_t *s_ha = S.head_a, *s_hb = S.head_b, *s_mix = S.mix, *s_df = S.df, *s_act = S.act;
    int *s_range = S.range;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t wid = win_list ? win_list[blockIdx.x] : blockIdx.x;
    const uint64_t win = (uint64_t)wid * kRefWindow;
    const uint64_t w0 = win >> 5;
    for (int i = tid; i < HW; i += kRefThreads) {
        const uint32_t h = head_cur[w0 + i];
        s_ha[i] = h;
        s_hb[i] = h;
        s_mix[i] = 0;
        if (!ORDER) {
            s_act[i] = 0;
            s_df[i] = diff_bits ? diff_bits[w0 + i] : 0u;
        }
    }
    __syncthreads();

    // Ownership of the CTA: the groups whose head lies in [win, win+kRefWindow).
    if (warp == 0) {
        const uint32_t hw = s_ha[lane];
        const uint32_t nz = __ballot_sync(0xffffffffu, hw != 0);
        int start = -1, end = -1;
        if (nz) {
            const int fl = __ffs(nz) - 1, ll = 31 - __clz(nz);
            const uint32_t fw = __shfl_sync(0xffffffffu, hw, fl), lw = __shfl_sync(0xffffffffu, hw, ll);
            start = fl * 32 + __ffs(fw) - 1;
            const int hl = ll * 32 + 31 - __clz(lw); // head of the last owned group
            const uint32_t ew = lane < OVER_WORDS ? s_ha[WIN_WORDS + lane] : 0u;
            const uint32_t enz = __ballot_sync(0xffffffffu, ew != 0);
            int e = -1;
            if (enz) {
                const int el = __ffs(enz) - 1;
                const uint32_t x = __shfl_sync(0xffffffffu, ew, el);
                e = kRefWindow + el * 32 + __ffs(x) - 1;
            }
            if (e >= 0 && e - hl <= kRwGroupMax) {
                end = e;
            } else {
                end = hl; // the last group is too large for shared memory: leave it to the global path
                if (lane == 0) {
                    const uint32_t slot = atomicAdd(big_count, 1u);
                    if (slot < big_cap) big_heads[slot] = (uint32_t)(win + hl);
                    // it comes back one depth deeper: this window is visited again
                    if (atomicExch(&win_flag[wid], 1u) == 0u) win_next[atomicAdd(win_next_count, 1u)] = wid;
                }
            }
        }
        if (lane == 0) {
            s_range[0] = start;
            s_range[1] = end;
        }
    }
    __syncthreads();
    const int start = s_range[0], end = s_range[1];
    if (start < 0 || end <= start) return;

    // this warp's slot range (`end` is a head, so the scan stops there at the latest)
    auto first_head_ge = [&](int x) -> int {
        if (x >= end) return end;
        int w = x >> 5;
        uint32_t m = s_ha[w] & (0xffffffffu << (x & 31));
        while (m == 0) m = s_ha[++w];
        const int q = (w << 5) + __ffs(m) - 1;
        return q < end ? q : end;
    };
    const int ws = first_head_ge(warp * PART);
    const int we = warp == NWARP - 1 ? end : first_head_ge((warp + 1) * PART);
    if (we <= ws) return;
    uint16_t *list = &S.list[ws];

    // keys of up to four suffixes per lane: all text words are requested before the first one is used
    auto fetch4 = [&](const uint64_t (&pos)[4], const int (&slot)[4], uint32_t dd) {
        uint64_t x0[4], x1[4];
        int sh[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (slot[u] >= 0) {
                const uint64_t q = pos[u] + dd;
                const uint64_t w = q / P::SPW;
                sh[u] = (int)(q - w * P::SPW);
                x0[u] = __ldg(packed + w);
                x1[u] = __ldg(packed + w + 1);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (slot[u] >= 0) s_key[slot[u]] = window_of<BITS>(x0[u], x1[u], sh[u]);
        }
    };

    // bits of this warp's range in head word i
    auto range_mask = [&](int i) -> uint32_t {
        const int lo = ws > (i << 5) ? ws - (i << 5) : 0, hi = (we - 1) - (i << 5) < 31 ? (we - 1) - (i << 5) : 31;
        return (0xffffffffu << lo) & (0xffffffffu >> (31 - hi));
    };
    auto mixed = [&](int g) -> bool { return (s_mix[g >> 5] >> (g & 31)) & 1u; };

    if (!ORDER) {
        // Which groups hold more than one BWT symbol.  After the initial sort the answer is in diff_bits (one
        // bit per slot whose symbol differs from its predecessor's in the same group, written by heads_kernel
        // while the symbols were in registers); later launches compare the bytes.
        if (diff_bits) {
            for (int i = (ws >> 5) + lane; i <= ((we - 1) >> 5); i += 32) {
                uint32_t dw = s_df[i] & range_mask(i);
                while (dw) {
                    const int g = prev_set_le(s_ha, (i << 5) + __ffs(dw) - 1);
                    dw &= dw - 1;
                    atomicOr(&s_mix[g >> 5], 1u << (g & 31));
                }
            }
        } else {
            for (int r = ws + lane; r < we; r += 32) {
                const bool h0 = (s_ha[r >> 5] >> (r & 31)) & 1u;
                const bool h1 = (s_ha[(r + 1) >> 5] >> ((r + 1) & 31)) & 1u;
                if (!(h0 && h1)) s_bw[0][r] = bwt[win + r];
            }
            __syncwarp();
            for (int r = ws + lane; r < we; r += 32) {
                const bool h0 = (s_ha[r >> 5] >> (r & 31)) & 1u;
                const bool h1 = (s_ha[(r + 1) >> 5] >> ((r + 1) & 31)) & 1u;
                if (!(h0 && h1) && !h0) { // a member behind its group's head
                    const int g = prev_set_le(s_ha, r);
                    if (s_bw[0][r] != s_bw[0][g]) atomicOr(&s_mix[g >> 5], 1u << (g & 31));
                }
            }
        }
        __syncwarp();
        // the slots of those groups
        for (int i = (ws >> 5) + lane; i <= ((we - 1) >> 5); i += 32) {
            uint32_t mw = s_mix[i] & range_mask(i);
            while (mw) {
                const int g = (i << 5) + __ffs(mw) - 1;
                mw &= mw - 1;
                const int e = next_set_gt(s_ha, g); // one behind the group's last slot
                for (int w = g >> 5; w <= (e - 1) >> 5; ++w) {
                    const int lo = g > (w << 5) ? g - (w << 5) : 0, hi = (e - 1) - (w << 5) < 31 ? (e - 1) - (w << 5) : 31;
                    atomicOr(&s_act[w], (0xffffffffu << lo) & (0xffffffffu >> (31 - hi)));
                }
            }
        }
        __syncwarp();
    }

    // load the suffixes (and their BWT bytes) that sit in groups that have to be sorted, and their first keys
    uint32_t d = depth;
    int cnt = 0;
    for (int b0 = ws; b0 < we; b0 += 128) {
        uint64_t pos[4];
        int slot[4];
        uint32_t sv[4];
        uint8_t bv[4], hv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { // the four loads of a lane are independent: issue them back to back
            const int r = b0 + u * 32 + lane;
            bool act = false;
            if (r < we) {
                const bool h0 = (s_ha[r >> 5] >> (r & 31)) & 1u;
                const bool h1 = (s_ha[(r + 1) >> 5] >> ((r + 1) & 31)) & 1u;
                act = ORDER ? !(h0 && h1) : ((s_act[r >> 5] >> (r & 31)) & 1u);
            }
            slot[u] = act ? r : -1;
            sv[u] = 0;
            bv[u] = hv[u] = 0;
            if (act) {
                sv[u] = sa[win + r];
                if (bwt) bv[u] = bwt[win + r];
                if (WIDE) hv[u] = sa_hi[win + r];
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int r = b0 + u * 32 + lane;
            const bool act = slot[u] >= 0;
            pos[u] = sv[u];
            if (act) {
                s_sa[0][r] = sv[u];
                s_bw[0][r] = bv[u];
                if (WIDE) {
                    s_hi[0][r] = hv[u];
                    pos[u] |= (uint64_t)hv[u] << lo_bits;
                }
            }
            const uint32_t m = __ballot_sync(0xffffffffu, act);
            if (act) list[cnt + __popc(m & lanemask_lt())] = (uint16_t)r;
            cnt += __popc(m);
        }
        fetch4(pos, slot, d);
    }
    __syncwarp();

    int c = 0;
    unsigned long long fetched = 0;
    // The ranking notes for every slot the first slot of the group it put the suffix in, which saves the steps after
    // it their bit scans.  It leaves the list alone: a group's members go to the group's own slots, so as a set of
    // slots -- all the later steps need -- the list is the same before and after, and it stays in slot order.
    uint16_t *ghead = S.ghead;
    while (cnt > 0) {
        fetched += (unsigned)cnt;
        // rank: stable position inside the group; a suffix opens a new group iff no earlier member
        // carries the same key (or its key holds the terminator, which makes it unique)
        int nbig = 0; // large groups of this warp's range seen in this step (warp-uniform)
        if (!COOP) {
            // Whole groups, as many as fit the 32 lanes, one member per lane.  The list holds whole groups in slot
            // order (it starts that way, and the classification below compacts it in order), so a group is a run of
            // lanes between two head flags; match.any finds the lanes that carry
            // a lane's key (its class), the count of earlier ones is its rank among equals, and the members with
            // smaller keys are counted class by class -- a group rarely holds more than a few distinct keys.
            for (int i0 = 0; i0 < cnt;) {
                const int i = i0 + lane;
                const bool valid = i < cnt;
                const int r = valid ? list[i] : 0;
                const uint32_t hb = __ballot_sync(0xffffffffu, valid && ((s_ha[r >> 5] >> (r & 31)) & 1u)) | 1u;
                int take = cnt - i0 < 32 ? cnt - i0 : 32;
                if (i0 + 32 < cnt) { // the group at the end of the window may go on behind it
                    const int rn = list[i0 + 32];
                    if (!((s_ha[rn >> 5] >> (rn & 31)) & 1u)) take = 31 - __clz(hb);
                }
                if (take == 0) {
                    // a group of more than 32 members: every member against all others
                    const int gs = list[i0];
                    const int ge = next_set_gt(s_ha, gs);
                    for (int ii = i0 + lane; ii < i0 + (ge - gs); ii += 32) {
                        const int rr = list[ii];
                        const uint64_t mk = s_key[rr];
                        int lt = 0, eq = 0;
                        for (int j = gs; j < ge; ++j) {
                            const uint64_t o = s_key[j];
                            lt += o < mk;
                            eq += (o == mk) & (j < rr);
                        }
                        const int p = gs + lt + eq;
                        if (p != gs && (eq == 0 || key_terminated<BITS>(mk))) atomicOr(&s_hb[p >> 5], 1u << (p & 31));
                        ghead[p] = (uint16_t)(key_terminated<BITS>(mk) ? p : gs + lt);
                        s_sa[c ^ 1][p] = s_sa[c][rr];
                        s_bw[c ^ 1][p] = s_bw[c][rr];
                        if (WIDE) s_hi[c ^ 1][p] = s_hi[c][rr];
                    }
                    i0 += ge - gs;
                    continue;
                }
                const bool in = lane < take;
                const uint32_t takemask = take >= 32 ? 0xffffffffu : ((1u << take) - 1);
                const uint32_t upto = 0xffffffffu >> (31 - lane);               // lanes <= this one
                const int sl = 31 - __clz(hb & upto);                            // lane of my group's head
                const uint32_t above = hb & ~upto & takemask;
                const int el = above ? __ffs(above) - 1 : take;                  // one behind my group's last lane
                const uint32_t gmask = (el >= 32 ? 0xffffffffu : ((1u << el) - 1)) & ~((1u << sl) - 1);
                const uint64_t mk = valid ? s_key[r] : 0ull;
                const uint32_t E = __match_any_sync(0xffffffffu, mk) & gmask;
                const int eq = __popc(E & lanemask_lt());
                int lt = 0;
                uint32_t rem = in ? (gmask & ~E) : 0u; // members of my group with other keys
                while (__any_sync(0xffffffffu, rem != 0)) {
                    const int l = rem ? __ffs(rem) - 1 : lane;
                    const uint64_t kl = __shfl_sync(0xffffffffu, mk, l);
                    const uint32_t El = __shfl_sync(0xffffffffu, E, l);
                    if (rem) {
                        if (kl < mk) lt += __popc(El);
                        rem &= ~El;
                    }
                }
                const int gs = __shfl_sync(0xffffffffu, r, sl);
                if (in) {
                    const int p = gs + lt + eq;
                    if (p != gs && (eq == 0 || key_terminated<BITS>(mk))) atomicOr(&s_hb[p >> 5], 1u << (p & 31));
                    ghead[p] = (uint16_t)(key_terminated<BITS>(mk) ? p : gs + lt); // the equal ones start at gs + lt
                    s_sa[c ^ 1][p] = s_sa[c][r];
                    s_bw[c ^ 1][p] = s_bw[c][r]; // the BWT symbol moves with its suffix
                    if (WIDE) s_hi[c ^ 1][p] = s_hi[c][r];
                    // (the list stays as it is: the group's members went to the group's slots, and the steps below
                    // only need the set of slots -- in slot order, which the next step's lane runs rely on)
                }
                i0 += take;
            }
        } else
        for (int i0 = 0; i0 < cnt; i0 += 32) {
            const int i = i0 + lane;
            bool big_first = false;
            int gs = 0;
            if (i < cnt) {
                const int r = list[i];
                gs = prev_set_le(s_ha, r);
                const int ge = next_set_gt(s_ha, r);
                if (ge - gs >= big_thr) {
                    big_first = r == gs; // the whole warp ranks this group below
                } else {
                    const uint64_t mk = s_key[r];
                    int lt = 0, eq = 0;
                    for (int j = gs; j < r; ++j) {
                        const uint64_t o = s_key[j];
                        lt += o < mk;
                        eq += o == mk;
                    }
                    for (int j = r + 1; j < ge; ++j) lt += s_key[j] < mk;
                    const int p = gs + lt + eq;
                    if (p != gs && (eq == 0 || key_terminated<BITS>(mk))) atomicOr(&s_hb[p >> 5], 1u << (p & 31));
                    ghead[p] = (uint16_t)(key_terminated<BITS>(mk) ? p : gs + lt);
                    s_sa[c ^ 1][p] = s_sa[c][r];
                    s_bw[c ^ 1][p] = s_bw[c][r]; // the BWT symbol moves with its suffix
                    if (WIDE) s_hi[c ^ 1][p] = s_hi[c][r];
                }
            }
            const uint32_t bm = __ballot_sync(0xffffffffu, big_first);
            if (big_first) S.bigq[warp][nbig + __popc(bm & lanemask_lt())] = (uint16_t)gs;
            nbig += __popc(bm);
        }
        __syncwarp();
        for (int q = 0; q < nbig; ++q) {
            const int gs = S.bigq[warp][q];
            const int ge = next_set_gt(s_ha, gs);
            const int g = ge - gs;
            // candidate for the dominant key: the member in the middle of the group
            const uint64_t ck = s_key[gs + (g >> 1)];
            __syncwarp();
            // pass 1: classes.  The members that do not carry the candidate key are compacted, in slot order, to
            // the front of the group's own key slots (a key is read by its lane before anything of its chunk is
            // written, and the write index never exceeds the read index), so that the ranking below reads dense keys.
            int n_lt = 0, n_eq = 0, n_nd = 0;
            for (int b0 = gs; b0 < ge; b0 += 32) {
                const int r = b0 + lane;
                const bool in = r < ge;
                uint64_t mk = 0;
                bool is_eq = false, is_lt = false;
                if (in) {
                    mk = s_key[r];
                    is_eq = mk == ck;
                    is_lt = mk < ck;
                }
                const uint32_t eqm = __ballot_sync(0xffffffffu, is_eq), ltm = __ballot_sync(0xffffffffu, is_lt);
                const uint32_t ndm = __ballot_sync(0xffffffffu, in && !is_eq);
                if (is_eq) S.newpos[r] = (uint16_t)(n_eq + __popc(eqm & lanemask_lt())); // rank among the equal ones
                if (in && !is_eq) {
                    const int t = gs + n_nd + __popc(ndm & lanemask_lt());
                    S.newpos[r] = 0xffffu; // not a carrier of the candidate key
                    S.nd[t] = (uint16_t)r;
                    s_key[t] = mk;
                }
                n_eq += __popc(eqm);
                n_lt += __popc(ltm);
                n_nd += __popc(ndm);
                __syncwarp();
            }
            // the carriers of the candidate key: their stable rank is their running count, no comparisons at all
            const bool term = key_terminated<BITS>(ck);
            for (int r = gs + lane; r < ge; r += 32) {
                const int e = S.newpos[r];
                if (e != 0xffff) {
                    const int p = gs + n_lt + e;
                    if (p != gs && (e == 0 || term)) atomicOr(&s_hb[p >> 5], 1u << (p & 31));
                    s_sa[c ^ 1][p] = s_sa[c][r];
                    s_bw[c ^ 1][p] = s_bw[c][r];
                    if (WIDE) s_hi[c ^ 1][p] = s_hi[c][r];
                    ghead[p] = (uint16_t)(term ? p : gs + n_lt);
                }
            }
            // the others against each other (dense keys in the first n_nd key slots of the group)
            for (int t = lane; t < n_nd; t += 32) {
                const int r = S.nd[gs + t];
                const uint64_t mk = s_key[gs + t];
                int lt = 0, eq = 0;
                for (int u = 0; u < n_nd; ++u) {
                    const uint64_t o = s_key[gs + u];
                    lt += o < mk;
                    eq += (o == mk) & (u < t);
                }
                const int p = gs + lt + eq + (mk > ck ? n_eq : 0);
                if (p != gs && (eq == 0 || key_terminated<BITS>(mk))) atomicOr(&s_hb[p >> 5], 1u << (p & 31));
                s_sa[c ^ 1][p] = s_sa[c][r];
                s_bw[c ^ 1][p] = s_bw[c][r];
                if (WIDE) s_hi[c ^ 1][p] = s_hi[c][r];
                ghead[p] = (uint16_t)(key_terminated<BITS>(mk) ? p : p - eq);
            }
            __syncwarp();
        }
        __syncwarp();
        if (!ORDER) {
            // which of the new groups still hold more than one BWT symbol
            for (int i = (ws >> 5) + lane; i <= ((we - 1) >> 5); i += 32) atomicAnd(&s_mix[i], ~range_mask(i));
            __syncwarp();
            for (int i = lane; i < cnt; i += 32) {
                const int p = list[i];
                const int g = ghead[p];
                if (g != p && s_bw[c ^ 1][p] != s_bw[c ^ 1][g]) atomicOr(&s_mix[g >> 5], 1u << (g & 31));
            }
            __syncwarp();
        }
        // classify: resolved suffixes go home now; the rest stay on the list (compacted in place: an entry
        // is written at or before the position it was read from, and a warp reads 32 entries before it writes)
        d += P::SPW;
        int next = 0;
        for (int i = lane; (i & ~31) < cnt; i += 32) {
            bool again = false;
            int p = 0;
            if (i < cnt) {
                p = list[i];
                const bool h0 = (s_hb[p >> 5] >> (p & 31)) & 1u;
                const bool h1 = (s_hb[(p + 1) >> 5] >> ((p + 1) & 31)) & 1u;
                again = !(h0 && h1);
                if (!ORDER && again) again = mixed(ghead[p]);
                if (!again) {
                    sa[win + p] = s_sa[c ^ 1][p];
                    if (bwt) bwt[win + p] = s_bw[c ^ 1][p];
                    if (WIDE) sa_hi[win + p] = s_hi[c ^ 1][p];
                }
            }
            const uint32_t m = __ballot_sync(0xffffffffu, again);
            if (again) list[next + __popc(m & lanemask_lt())] = (uint16_t)p;
            next += __popc(m);
        }
        __syncwarp();
        // next keys of the survivors
        for (int i0 = lane; (i0 & ~31) < next; i0 += 128) {
            uint64_t pos[4];
            int slot[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * 32;
                slot[u] = -1;
                pos[u] = 0;
                if (i < next) {
                    const int p = list[i];
                    slot[u] = p;
                    pos[u] = WIDE ? (((uint64_t)s_hi[c ^ 1][p] << lo_bits) | s_sa[c ^ 1][p]) : (uint64_t)s_sa[c ^ 1][p];
                }
            }
            fetch4(pos, slot, d);
        }
        // publish the new heads of this range (bits only ever get set; neighbours' bits are left alone)
        for (int i = (ws >> 5) + lane; i <= ((we - 1) >> 5); i += 32) {
            const uint32_t add = s_hb[i] & range_mask(i) & ~s_ha[i];
            if (add) atomicOr(&s_ha[i], add);
        }
        c ^= 1;
        cnt = next;
        __syncwarp();
    }

    for (int i = (ws >> 5) + lane; i <= ((we - 1) >> 5); i += 32) {
        const uint32_t fresh = s_hb[i] & ~head_cur[w0 + i];
        if (fresh) atomicOr(&head_next[w0 + i], fresh);
    }
    if (lane == 0 && fetched) atomicAdd(&remaining[64 + ((wid + warp) & 63)], fetched);
}

// ---------------------------------------------------------------------------
// compaction of the groups that have to be sorted
// ---------------------------------------------------------------------------
// When only the BWT is wanted, most tie groups need no sorting (see refine_warps_kernel, ORDER = false) and
// a refinement that visits every window of the suffix array spends its time finding out that there is
// little to do.  The groups with mixed BWT symbols are therefore copied out first, in order, into dense
// arrays (suffix, BWT byte, high position byte, original slot, group heads); the refinement runs on those
// as on a much shorter suffix array, and only the BWT bytes are copied back to their slots afterwards.
constexpr int kActTileWords = 256; // head words per CTA in the compaction passes (8192 slots)

// act bit i = slot i belongs to a group holding a diff bit; act is zeroed by the caller.
// word t of the difference bitmap: every group that holds one of its bits is marked from its head to its last slot
__device__ __forceinline__ void mark_word(const uint32_t *__restrict__ head, uint64_t t, uint32_t dw, uint32_t *__restrict__ act)
{
    uint64_t done_to = 0; // slots below this are already marked by this thread
    while (dw) {
        const int b = __ffs(dw) - 1;
        dw &= dw - 1;
        const uint64_t slot = t * 32 + b;
        if (slot < done_to) continue; // same group as the previous diff bit
        // group head: last head bit at or before slot (a diff bit is never a head itself)
        uint64_t w = t;
        uint32_t m = head[w] & (0xffffffffu >> (31 - b));
        while (m == 0) m = head[--w];
        const uint64_t g = w * 32 + (31 - __clz(m));
        // one behind its last slot: first head bit after slot
        w = t;
        m = b == 31 ? 0u : (head[w] & (0xffffffffu << (b + 1)));
        while (m == 0) m = head[++w];
        const uint64_t e = w * 32 + (__ffs(m) - 1);
        for (uint64_t x = g >> 5; x <= (e - 1) >> 5; ++x) {
            const int lo = g > (x << 5) ? (int)(g - (x << 5)) : 0;
            const int hi = (e - 1) - (x << 5) < 31 ? (int)((e - 1) - (x << 5)) : 31;
            atomicOr(&act[x], (0xffffffffu << lo) & (0xffffffffu >> (31 - hi)));
        }
        done_to = e;
    }
}

// four words of the difference bitmap per thread, fetched as one 16-byte load (most of them are zero)
__global__ void __launch_bounds__(256) mark_active_kernel(const uint32_t *__restrict__ head, const uint32_t *__restrict__ diff,
                                                          uint64_t nwords, uint32_t *__restrict__ act)
{
    const uint64_t t0 = ((uint64_t)blockIdx.x * 256 + threadIdx.x) * 4;
    if (t0 >= nwords) return;
    uint32_t dv[4] = {0u, 0u, 0u, 0u};
    if (t0 + 4 <= nwords) {
        const uint4 x = *reinterpret_cast<const uint4 *>(diff + t0);
        dv[0] = x.x; dv[1] = x.y; dv[2] = x.z; dv[3] = x.w;
    } else {
        for (int u = 0; u < 4; ++u)
            if (t0 + u < nwords) dv[u] = diff[t0 + u];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
        if (dv[u]) mark_word(head, t0 + u, dv[u], act);
}

__global__ void __launch_bounds__(256) count_active_kernel(const uint32_t *__restrict__ act, uint64_t nwords,
                                                           uint64_t *__restrict__ tile_count)
{
    __shared__ uint32_t s_w[8];
    const uint64_t t = (uint64_t)blockIdx.x * kActTileWords + threadIdx.x;
    uint32_t c = t < nwords ? __popc(act[t]) : 0u;
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int k = 0; k < 8; ++k) tot += s_w[k];
        tile_count[blockIdx.x] = tot;
    }
}

// exclusive scan of u64 counts in place, total behind the last entry; one block, eight consecutive entries per thread
__global__ void __launch_bounds__(1024) scan_tiles_kernel(uint64_t *__restrict__ v, uint64_t n)
{
    constexpr int ITEMS = 8;
    __shared__ uint64_t scratch[33];
    uint64_t carry = 0;
    for (uint64_t base = 0; base < n; base += 1024 * ITEMS) {
        const uint64_t i0 = base + (uint64_t)threadIdx.x * ITEMS;
        uint64_t x[ITEMS], sum = 0;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            x[k] = i0 + k < n ? v[i0 + k] : 0;
            sum += x[k];
        }
        uint64_t total;
        uint64_t e = carry + block_excl_sum(sum, scratch, &total);
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            if (i0 + k < n) v[i0 + k] = e;
            e += x[k];
        }
        carry += total;
    }
    if (threadIdx.x == 0) v[n] = carry;
}

// The active slots, in order, into dense arrays.  chead must be zeroed; its bit j is set iff compact entry j
// starts a group, and every bit from m_act on is set (what heads_kernel does behind the last suffix).
__global__ void __launch_bounds__(256)
compact_active_kernel(const uint32_t *__restrict__ act, const uint32_t *__restrict__ head, uint64_t nwords,
                      const uint64_t *__restrict__ tile_off, const uint32_t *__restrict__ sa, const uint8_t *__restrict__ bwt,
                      const uint8_t *__restrict__ sa_hi, uint32_t *__restrict__ csa, uint8_t *__restrict__ cbw,
                      uint8_t *__restrict__ chi, uint32_t *__restrict__ corig, uint32_t *__restrict__ chead)
{
    // A warp owns 32 words (1024 slots) of the tile.  Its active slots are handled 32 at a time, one per lane and in
    // order: the lane finds the word of its slot in the warp's prefix sums (five shuffles), the bit inside the word
    // (find-nth-set), and copies -- reads that follow the runs of active slots, writes that are dense.
    __shared__ uint32_t scratch[9];
    const int lane = threadIdx.x & 31;
    const uint64_t t = (uint64_t)blockIdx.x * kActTileWords + threadIdx.x;
    const uint32_t a = t < nwords ? act[t] : 0u;
    const uint32_t hd = t < nwords ? head[t] : 0u;
    const uint32_t c = __popc(a);
    uint32_t total;
    const uint32_t e = block_excl_sum(c, scratch, &total);
    const uint32_t ex = e - __shfl_sync(0xffffffffu, e, 0);           // active slots of the warp's words in front of mine
    const uint32_t T = __shfl_sync(0xffffffffu, ex + c, 31);          // active slots of the warp
    if (T == 0) return;
    const uint64_t j0 = tile_off[blockIdx.x] + __shfl_sync(0xffffffffu, e, 0); // dense index of the warp's first active slot
    const uint64_t word0 = t - lane;
    for (uint32_t k0 = 0; k0 < T; k0 += 32) {
        const uint32_t k = k0 + lane;
        const bool valid = k < T;
        // the last word whose prefix does not exceed k holds the k-th active slot
        int L = 0;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
            const uint32_t ec = __shfl_sync(0xffffffffu, ex, (L + step) & 31);
            if (L + step < 32 && ec <= k) L += step;
        }
        const uint32_t aL = __shfl_sync(0xffffffffu, a, L);
        const uint32_t hL = __shfl_sync(0xffffffffu, hd, L);
        const uint32_t exL = __shfl_sync(0xffffffffu, ex, L);
        bool hbit = false;
        if (valid) {
            const int b = (int)__fns(aL, 0, (int)(k - exL) + 1);
            const uint64_t slot = (word0 + L) * 32 + b;
            const uint64_t j = j0 + k;
            hbit = (hL >> b) & 1u;
            csa[j] = sa[slot];
            cbw[j] = bwt[slot];
            if (chi) chi[j] = sa_hi[slot];
            corig[j] = (uint32_t)slot;
        }
        // head bits of these 32 entries, at bit offset j0 + k0 of chead (words shared with the neighbours: OR)
        const uint32_t hbm = __ballot_sync(0xffffffffu, hbit);
        const uint64_t o = j0 + k0;
        const int sh = (int)(o & 31);
        if (lane == 0 && (hbm << sh)) atomicOr(&chead[o >> 5], hbm << sh);
        if (lane == 1 && sh && (hbm >> (32 - sh))) atomicOr(&chead[(o >> 5) + 1], hbm >> (32 - sh));
    }
}

// bits m_act.. of the compact head bitmap (head_words words)
__global__ void __launch_bounds__(256) pad_heads_kernel(uint32_t *__restrict__ chead, uint64_t m_act, uint64_t head_words)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t w = (m_act >> 5) + (uint64_t)blockIdx.x * 256 + threadIdx.x; w < head_words; w += stride) {
        if (w == (m_act >> 5))
            atomicOr(&chead[w], 0xffffffffu << (m_act & 31));
        else
            chead[w] = 0xffffffffu;
    }
}

// BWT bytes of the compact entries back to their slots
__global__ void __launch_bounds__(256) scatter_bwt_kernel(const uint32_t *__restrict__ corig, const uint8_t *__restrict__ cbw,
                                                          uint64_t m_act, uint8_t *__restrict__ bwt)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x; j < m_act; j += stride) bwt[corig[j]] = cbw[j];
}

// ---------------------------------------------------------------------------
// large-group path
// ---------------------------------------------------------------------------
// One warp per listed group: distance from its head to the next head.
__global__ void __launch_bounds__(256) big_extent_kernel(const uint32_t *__restrict__ head_cur, uint64_t n,
                                                         const uint32_t *__restrict__ big_heads, uint32_t nbig,
                                                         uint32_t *__restrict__ big_len)
{
    const int lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (g >= nbig) return;
    const uint64_t h = big_heads[g];
    // first set bit at a position > h (bits >= n are set, so the scan ends)
    uint64_t w = h >> 5;
    uint32_t first = (h & 31) == 31 ? 0u : (head_cur[w] & (0xffffffffu << ((h & 31) + 1)));
    uint64_t found = ~0ull;
    if (first) {
        found = (w << 5) + __ffs(first) - 1;
    } else {
        for (uint64_t base = w + 1;; base += 32) {
            const uint32_t x = head_cur[base + lane];
            const uint32_t nz = __ballot_sync(0xffffffffu, x != 0);
            if (nz) {
                const int l = __ffs(nz) - 1;
                const uint32_t xw = __shfl_sync(0xffffffffu, x, l);
                found = ((base + l) << 5) + __ffs(xw) - 1;
                break;
            }
        }
    }
    if (found > n) found = n;
    if (lane == 0) big_len[g] = (uint32_t)(found - h);
}

__device__ __forceinline__ uint32_t find_group(const uint64_t *__restrict__ off, uint32_t nbig, uint64_t j)
{
    // largest g with off[g] <= j  (off has nbig+1 entries, off[nbig] = total)
    uint32_t lo = 0, hi = nbig;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (off[mid] <= j) lo = mid; else hi = mid;
    }
    return lo;
}

template <int BITS>
__global__ void __launch_bounds__(256)
big_gather_kernel(const uint64_t *__restrict__ packed, const uint32_t *__restrict__ sa, uint32_t depth,
                  const uint32_t *__restrict__ big_heads, const uint64_t *__restrict__ big_off, uint32_t nbig,
                  uint64_t total, uint32_t *__restrict__ bsa, uint64_t *__restrict__ bkey, uint32_t *__restrict__ bgid,
                  const uint8_t *__restrict__ sa_hi, uint8_t *__restrict__ bhi, int lo_bits)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x; j < total; j += stride) {
        const uint32_t g = find_group(big_off, nbig, j);
        const uint64_t slot = (uint64_t)big_heads[g] + (j - big_off[g]);
        const uint32_t s = sa[slot];
        uint64_t pos = s;
        if (sa_hi) {
            const uint8_t h = sa_hi[slot];
            bhi[j] = h;
            pos |= (uint64_t)h << lo_bits;
        }
        bsa[j] = s;
        bkey[j] = text_window<BITS>(packed, pos + depth);
        bgid[j] = g;
    }
}

__global__ void __launch_bounds__(256) gather_u32_to_u64_kernel(const uint32_t *__restrict__ src,
                                                                const uint32_t *__restrict__ perm, uint64_t n,
                                                                uint64_t *__restrict__ dst)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x; j < n; j += stride) dst[j] = src[perm[j]];
}

template <int BITS>
__global__ void __launch_bounds__(256)
big_scatter_kernel(const uint32_t *__restrict__ perm, const uint32_t *__restrict__ bsa,
                   const uint64_t *__restrict__ bkey, const uint32_t *__restrict__ bgid,
                   const uint32_t *__restrict__ big_heads, const uint64_t *__restrict__ big_off, uint64_t total,
                   uint32_t *__restrict__ sa, uint32_t *__restrict__ head_next, uint32_t *__restrict__ win_flag,
                   uint32_t *__restrict__ win_next, uint32_t *__restrict__ win_next_count,
                   const uint64_t *__restrict__ packed, const uint8_t *__restrict__ inv_map, uint8_t *__restrict__ bwt,
                   const uint8_t *__restrict__ bhi, uint8_t *__restrict__ sa_hi, int lo_bits)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x; j < total; j += stride) {
        const uint32_t idx = perm[j];
        const uint32_t g = bgid[idx];
        const uint64_t slot = (uint64_t)big_heads[g] + (j - big_off[g]);
        const uint32_t plo = bsa[idx];
        uint64_t pos = plo;
        if (sa_hi) {
            const uint8_t h = bhi[idx];
            sa_hi[slot] = h;
            pos |= (uint64_t)h << lo_bits;
        }
        sa[slot] = plo;
        if (bwt) bwt[slot] = pos ? inv_map[text_symbol<BITS>(packed, pos - 1)] : 0;
        // every window under a re-sorted large group is looked at again in the next round
        const uint32_t wnd = (uint32_t)(slot / kRefWindow);
        if (win_flag[wnd] == 0u && atomicExch(&win_flag[wnd], 1u) == 0u) win_next[atomicAdd(win_next_count, 1u)] = wnd;
        if (j > big_off[g]) {
            const uint64_t me = bkey[idx], before = bkey[perm[j - 1]];
            if (key_terminated<BITS>(me) || me != before) atomicOr(&head_next[slot >> 5], 1u << (slot & 31));
        }
    }
}

// text positions as u64: hi << lo_bits | lo  (export of a slice of a wide build)
__global__ void __launch_bounds__(256) widen_sa_kernel(const uint32_t *__restrict__ lo, const uint8_t *__restrict__ hi,
                                                       int lo_bits, uint64_t n, uint64_t *__restrict__ out)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride)
        out[i] = (hi ? ((uint64_t)hi[i] << lo_bits) : 0ull) | lo[i];
}

// ---------------------------------------------------------------------------
// BWT
// ---------------------------------------------------------------------------
// bwt[i] = byte of the symbol before suffix i (0 for a whole document).  The symbol is gathered from the
// packed text (3/8 of the raw text's footprint) and mapped back to its byte through `inv_map`.
template <int BITS>
__global__ void __launch_bounds__(256) bwt_kernel(const uint64_t *__restrict__ packed,
                                                  const uint8_t *__restrict__ inv_map,
                                                  const uint32_t *__restrict__ sa, uint64_t n,
                                                  uint8_t *__restrict__ bwt)
{
    __shared__ uint8_t s_inv[256];
    s_inv[threadIdx.x] = inv_map[threadIdx.x];
    __syncthreads();
    const uint64_t noct = n / 8;
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x; q < noct; q += stride) {
        const uint4 a = *reinterpret_cast<const uint4 *>(sa + 8 * q);
        const uint4 b = *reinterpret_cast<const uint4 *>(sa + 8 * q + 4);
        const uint32_t p[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t c[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) c[j] = p[j] ? text_symbol<BITS>(packed, (uint64_t)p[j] - 1) : 0u;
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            lo |= (uint32_t)s_inv[c[j]] << (8 * j);
            hi |= (uint32_t)s_inv[c[4 + j]] << (8 * j);
        }
        *reinterpret_cast<uint2 *>(bwt + 8 * q) = make_uint2(lo, hi);
    }
    if (blockIdx.x == 0)
        for (uint64_t i = noct * 8 + threadIdx.x; i < n; i += 256) {
            const uint32_t p = sa[i];
            bwt[i] = p ? s_inv[text_symbol<BITS>(packed, (uint64_t)p - 1)] : 0;
        }
}

// ---------------------------------------------------------------------------
// suffix-array samples (the reference's dormant FMIndex::maketables, FMIndex.cpp:572-714)
// ---------------------------------------------------------------------------
constexpr int kTermTile = 4096; // raw bytes per CTA (256 threads x 16)

// terminators per tile / their positions in text order (document k ends at doc_end[k])
__global__ void __launch_bounds__(256) term_count_kernel(const uint8_t *__restrict__ raw, uint64_t n,
                                                         uint64_t *__restrict__ tile_count)
{
    __shared__ uint32_t s_sum[8];
    const uint64_t p0 = (uint64_t)blockIdx.x * kTermTile + (uint64_t)threadIdx.x * 16;
    uint32_t c = 0;
    for (int j = 0; j < 16; ++j)
        if (p0 + j < n) c += raw[p0 + j] == 0;
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int k = 0; k < 8; ++k) t += s_sum[k];
        tile_count[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) term_write_kernel(const uint8_t *__restrict__ raw, uint64_t n,
                                                         const uint64_t *__restrict__ tile_off,
                                                         uint32_t *__restrict__ doc_end)
{
    __shared__ uint32_t scratch[9];
    const uint64_t p0 = (uint64_t)blockIdx.x * kTermTile + (uint64_t)threadIdx.x * 16;
    uint32_t mask = 0;
    for (int j = 0; j < 16; ++j)
        if (p0 + j < n && raw[p0 + j] == 0) mask |= 1u << j;
    uint32_t total;
    uint64_t o = tile_off[blockIdx.x] + block_excl_sum((uint32_t)__popc(mask), scratch, &total);
    while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        doc_end[o++] = (uint32_t)(p0 + j);
    }
}

// FMIndex.cpp:624: the suffix at text position x = i+1 is sampled iff (end marker of its document - i) is a
// positive multiple of the sample rate and i lies in the same document.  One thread per document marks them
// in a bitmap indexed by text position.
__global__ void __launch_bounds__(256) sa_mark_kernel(const uint32_t *__restrict__ doc_end, uint32_t ndocs,
                                                      uint32_t rate, uint32_t *__restrict__ mark)
{
    const uint32_t k = blockIdx.x * 256 + threadIdx.x;
    if (k >= ndocs) return;
    const int64_t e = doc_end[k], s = k ? (int64_t)doc_end[k - 1] + 1 : 0;
    for (int64_t i = e - rate; i >= s; i -= rate) {
        const uint64_t x = (uint64_t)i + 1;
        atomicOr(&mark[x >> 5], 1u << (x & 31));
    }
}

// bit p of `out` (rank order) = mark[sa[p]] (by_mark) or bwt[p] == 0
__global__ void __launch_bounds__(256) sa_rank_bits_kernel(const uint32_t *__restrict__ sa, const uint8_t *__restrict__ bwt,
                                                           const uint32_t *__restrict__ mark, uint64_t n,
                                                           uint32_t *__restrict__ out, uint64_t out_words)
{
    const int lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * 8;
    for (uint64_t w = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); w < out_words; w += warps) {
        const uint64_t p = w * 32 + lane;
        bool bit = false;
        if (p < n) {
            if (mark) {
                const uint32_t x = sa[p];
                bit = (mark[x >> 5] >> (x & 31)) & 1u;
            } else {
                bit = bwt[p] == 0;
            }
        }
        const uint32_t word = __ballot_sync(0xffffffffu, bit);
        if (lane == 0) out[w] = word;
    }
}

// For every set bit p of `bits` (with its BitRank directories): j = rank1(p) - 1; doc = document holding text
// position sa[p]; out_doc[j] = doc; out_off[j] = sa[p] - start of doc  (FMIndex.cpp:676-699, 636-637).
__global__ void __launch_bounds__(256) sa_emit_kernel(const uint32_t *__restrict__ sa, const uint64_t *__restrict__ bits,
                                                      const uint64_t *__restrict__ Rs, const uint8_t *__restrict__ Rb,
                                                      uint64_t n, const uint32_t *__restrict__ doc_end, uint32_t ndocs,
                                                      uint32_t *__restrict__ out_doc, uint32_t *__restrict__ out_off)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x; p < n; p += stride) {
        const uint64_t word = bits[p >> 6];
        if (!((word >> (p & 63)) & 1ull)) continue;
        const uint64_t j = Rs[p >> 8] + Rb[p >> 6] + __popcll(word & ((1ull << (p & 63)) - 1)); // ones before p
        const uint32_t x = sa[p];
        uint32_t lo = 0, hi = ndocs - 1; // first document whose end marker is at or after x
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (doc_end[mid] >= x) hi = mid; else lo = mid + 1;
        }
        out_doc[j] = lo;
        if (out_off) out_off[j] = x - (lo ? doc_end[lo - 1] + 1 : 0u);
    }
}

// ---- the same over one slice of a packed-text build: u64 positions in the padded text ----
// Slot s holds geom.bytes[s] real symbols from position s * slot_syms on, then code-0 padding that must not read as
// terminators.  slot_syms is a multiple of 16 (whole 16-word lines of slots), so the 16 positions of one thread lie
// in one slot.
template <int BITS>
__device__ __forceinline__ uint32_t packed_term_mask(const uint64_t *__restrict__ packed, uint64_t n_text, const SelGeom &g,
                                                     uint64_t p0)
{
    using P = Pack<BITS>;
    const uint64_t slot_syms = g.slot_words * P::SPW;
    if (p0 >= n_text) return 0;
    const uint64_t s = p0 / slot_syms, in = p0 - s * slot_syms;
    const uint64_t real = g.bytes[s] > in ? g.bytes[s] - in : 0;
    uint32_t mask = 0;
    for (int j = 0; j < 16 && (uint64_t)j < real; ++j)
        if (text_symbol<BITS>(packed, p0 + j) == 0) mask |= 1u << j;
    return mask;
}

template <int BITS>
__global__ void __launch_bounds__(256) packed_term_count_kernel(const uint64_t *__restrict__ packed, uint64_t n_text,
                                                                const SelGeom g, uint64_t *__restrict__ tile_count)
{
    __shared__ uint32_t s_sum[8];
    const uint64_t p0 = (uint64_t)blockIdx.x * kTermTile + (uint64_t)threadIdx.x * 16;
    uint32_t c = (uint32_t)__popc(packed_term_mask<BITS>(packed, n_text, g, p0));
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int k = 0; k < 8; ++k) t += s_sum[k];
        tile_count[blockIdx.x] = t;
    }
}

template <int BITS>
__global__ void __launch_bounds__(256) packed_term_write_kernel(const uint64_t *__restrict__ packed, uint64_t n_text,
                                                                const SelGeom g, const uint64_t *__restrict__ tile_off,
                                                                uint64_t *__restrict__ doc_end)
{
    __shared__ uint32_t scratch[9];
    const uint64_t p0 = (uint64_t)blockIdx.x * kTermTile + (uint64_t)threadIdx.x * 16;
    uint32_t mask = packed_term_mask<BITS>(packed, n_text, g, p0);
    uint32_t total;
    uint64_t o = tile_off[blockIdx.x] + block_excl_sum((uint32_t)__popc(mask), scratch, &total);
    while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        doc_end[o++] = p0 + j;
    }
}

// first position of document k: one past the previous terminator, or the first symbol of k's slot
__device__ __forceinline__ uint64_t padded_doc_start(const uint64_t *__restrict__ doc_end, uint64_t k, uint64_t slot_syms)
{
    const uint64_t e = doc_end[k], slot_begin = e - e % slot_syms;
    const uint64_t after_prev = k ? doc_end[k - 1] + 1 : 0;
    return after_prev > slot_begin ? after_prev : slot_begin;
}

// sa_mark_kernel on padded positions
__global__ void __launch_bounds__(256) sa_mark64_kernel(const uint64_t *__restrict__ doc_end, uint32_t ndocs, uint32_t rate,
                                                        uint64_t slot_syms, uint32_t *__restrict__ mark)
{
    const uint64_t k = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (k >= ndocs) return;
    const uint64_t e = doc_end[k], s = padded_doc_start(doc_end, k, slot_syms);
    for (uint64_t d = rate; d <= e - s; d += rate) { // i = e - d >= s
        const uint64_t x = e - d + 1;
        atomicOr(&mark[x >> 5], 1u << (x & 31));
    }
}

__device__ __forceinline__ uint64_t slice_position(const uint32_t *__restrict__ sa, const uint8_t *__restrict__ hi, int lo_bits,
                                                   uint64_t p)
{
    return hi ? ((uint64_t)hi[p] << lo_bits) | sa[p] : (uint64_t)sa[p];
}

__global__ void __launch_bounds__(256) sa_slice_bits_kernel(const uint32_t *__restrict__ sa, const uint8_t *__restrict__ hi,
                                                            int lo_bits, const uint8_t *__restrict__ bwt,
                                                            const uint32_t *__restrict__ mark, uint64_t m,
                                                            uint32_t *__restrict__ sampled, uint64_t sampled_base,
                                                            uint32_t *__restrict__ ends, unsigned long long *__restrict__ counts)
{
    const int lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * 8, out_words = (m + 31) / 32;
    const uint64_t w0 = sampled_base >> 5;
    const int sh = (int)(sampled_base & 31);
    uint32_t n_s = 0, n_e = 0;
    for (uint64_t w = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); w < out_words; w += warps) {
        const uint64_t p = w * 32 + lane;
        bool bs = false, be = false;
        if (p < m) {
            const uint64_t x = slice_position(sa, hi, lo_bits, p);
            bs = (mark[x >> 5] >> (x & 31)) & 1u;
            be = bwt[p] == 0;
        }
        const uint32_t ws = __ballot_sync(0xffffffffu, bs), we = __ballot_sync(0xffffffffu, be);
        if (lane == 0) {
            ends[w] = we;
            // neighbouring warps share the boundary words of the shifted slice
            if (ws) {
                atomicOr(&sampled[w0 + w], ws << sh);
                if (sh && (ws >> (32 - sh))) atomicOr(&sampled[w0 + w + 1], ws >> (32 - sh));
            }
            n_s += (uint32_t)__popc(ws);
            n_e += (uint32_t)__popc(we);
        }
    }
    if (lane == 0) {
        if (n_s) atomicAdd(&counts[0], (unsigned long long)n_s);
        if (n_e) atomicAdd(&counts[1], (unsigned long long)n_e);
    }
}

// ORs a w-bit field (w <= 64) into a zeroed bit array, LSB first (Tools.h:49-61)
__device__ __forceinline__ void or_field(uint64_t *__restrict__ a, uint64_t bit, unsigned w, uint64_t v)
{
    if (w == 0) return;
    unsigned long long *p = reinterpret_cast<unsigned long long *>(a) + (bit >> 6);
    const unsigned sh = (unsigned)(bit & 63);
    atomicOr(p, (unsigned long long)(v << sh));
    if (sh + w > 64) atomicOr(p + 1, (unsigned long long)(v >> (64 - sh)));
}

__global__ void __launch_bounds__(256) sa_emit64_kernel(const uint32_t *__restrict__ sa, const uint8_t *__restrict__ hi,
                                                        int lo_bits, const uint64_t *__restrict__ bits,
                                                        const uint64_t *__restrict__ Rs, const uint8_t *__restrict__ Rb,
                                                        uint64_t bits_base, uint64_t rank_sub, uint64_t m,
                                                        const uint64_t *__restrict__ doc_end, uint32_t ndocs, uint64_t slot_syms,
                                                        uint64_t *__restrict__ doc_out, uint64_t doc_bit0, unsigned doc_w,
                                                        uint64_t *__restrict__ off_out, uint64_t off_bit0, unsigned off_w)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x; p < m; p += stride) {
        const uint64_t q = bits_base + p, word = bits[q >> 6];
        if (!((word >> (q & 63)) & 1ull)) continue;
        const uint64_t j = Rs[q >> 8] + Rb[q >> 6] + __popcll(word & ((1ull << (q & 63)) - 1)) - rank_sub;
        const uint64_t x = slice_position(sa, hi, lo_bits, p);
        uint32_t lo = 0, hi_d = ndocs - 1; // first document whose end marker is at or after x
        while (lo < hi_d) {
            const uint32_t mid = lo + (hi_d - lo) / 2;
            if (doc_end[mid] >= x) hi_d = mid; else lo = mid + 1;
        }
        or_field(doc_out, doc_bit0 + j * doc_w, doc_w, lo);
        if (off_out) or_field(off_out, off_bit0 + j * off_w, off_w, x - padded_doc_start(doc_end, lo, slot_syms));
    }
}

__global__ void __launch_bounds__(256) sa_lengths_kernel(const uint64_t *__restrict__ doc_end, uint64_t first, uint64_t count,
                                                         uint64_t slot_syms, uint64_t *__restrict__ out, uint64_t bit0,
                                                         unsigned w)
{
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t k = (uint64_t)blockIdx.x * 256 + threadIdx.x; k < count; k += stride) {
        const uint64_t g = first + k;
        or_field(out, bit0 + k * w, w, doc_end[g] - padded_doc_start(doc_end, g, slot_syms));
    }
}

// ---------------------------------------------------------------------------
// wavelet tree
// ---------------------------------------------------------------------------
constexpr int kWtInfoSmemNodes = 64; // node tables of up to this many internal nodes are staged in shared memory

// the 32 symbols of thread t of tile `tile`
__device__ __forceinline__ void wt_load32(const uint8_t *__restrict__ seq, uint64_t n, uint64_t p0, uint32_t (&w)[8])
{
    if (p0 + 32 <= n) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(seq + p0));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(seq + p0 + 16));
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
        w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            uint32_t x = 0;
            for (int j = 0; j < 4; ++j) {
                const uint64_t p = p0 + 4 * i + j;
                if (p < n) x |= (uint32_t)seq[p] << (8 * j);
            }
            w[i] = x;
        }
    }
}

// member / branch masks of the thread's 32 symbols for node table `info`
__device__ __forceinline__ void wt_masks(const uint8_t *info, const uint32_t (&w)[8], uint32_t valid, uint32_t &m,
                                         uint32_t &b)
{
    m = 0;
    b = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t v = info[(w[i] >> (8 * j)) & 0xff];
            m |= (v & 1u) << (4 * i + j);
            b |= (v >> 1) << (4 * i + j);
        }
    }
    m &= valid;
    b &= valid;
}

__device__ __forceinline__ uint32_t wt_valid_mask(uint64_t n, uint64_t p0)
{
    if (p0 >= n) return 0u;
    const uint64_t left = n - p0;
    return left >= 32 ? 0xffffffffu : ((1u << left) - 1u);
}

// Trees with at most 8 internal nodes (reads: 6): one table lookup per symbol yields its membership and branch
// bit for every node at once (low byte: member of node v, high byte: branch taken there); the bytes of eight symbols
// form an 8x8 bit matrix whose transpose holds every node's bits of those symbols (wt_masks_group) -- instead of
// one lookup per (symbol, node).
constexpr int kWtSmallNodes = 8;

__device__ __forceinline__ void wt_small_table(const uint8_t *__restrict__ node_info, int n_internal, uint16_t *lut16)
{
    uint32_t e = 0;
    for (int v = 0; v < n_internal; ++v) {
        const uint32_t x = node_info[v * 256 + threadIdx.x];
        e |= (x & 1u) << v;
        e |= ((x >> 1) & 1u) << (8 + v);
    }
    lut16[threadIdx.x] = (uint16_t)e;
}

// 8x8 bit matrix in two words (byte s = row s, rows 0..3 in lo), transposed in place: afterwards bit s of byte v is
// what bit v of byte s was (Hacker's Delight 7-3, on 32-bit halves: only the last step crosses the halves)
__device__ __forceinline__ void transpose8x8(uint32_t &lo, uint32_t &hi)
{
    uint32_t t;
    t = (lo ^ (lo >> 7)) & 0x00AA00AAu;
    lo ^= t ^ (t << 7);
    t = (hi ^ (hi >> 7)) & 0x00AA00AAu;
    hi ^= t ^ (t << 7);
    t = (lo ^ (lo >> 14)) & 0x0000CCCCu;
    lo ^= t ^ (t << 14);
    t = (hi ^ (hi >> 14)) & 0x0000CCCCu;
    hi ^= t ^ (t << 14);
    t = (lo ^ ((lo >> 28) | (hi << 4))) & 0xF0F0F0F0u;
    lo ^= t ^ (t << 28);
    hi ^= t >> 4;
}

// byte (V & 3) of src into byte G of dst
template <int G, int V> __device__ __forceinline__ uint32_t put_byte(uint32_t dst, uint32_t src)
{
    constexpr uint32_t sel = (0x3210u & ~(0xfu << (4 * G))) | ((4u + (V & 3)) << (4 * G));
    return __byte_perm(dst, src, sel);
}

template <int G>
__device__ __forceinline__ void wt_put_group(uint32_t lo, uint32_t hi, int n_internal, uint32_t (&out)[kWtSmallNodes])
{
    out[0] = put_byte<G, 0>(out[0], lo);
    if (1 < n_internal) out[1] = put_byte<G, 1>(out[1], lo);
    if (2 < n_internal) out[2] = put_byte<G, 2>(out[2], lo);
    if (3 < n_internal) out[3] = put_byte<G, 3>(out[3], lo);
    if (4 < n_internal) out[4] = put_byte<G, 4>(out[4], hi);
    if (5 < n_internal) out[5] = put_byte<G, 5>(out[5], hi);
    if (6 < n_internal) out[6] = put_byte<G, 6>(out[6], hi);
    if (7 < n_internal) out[7] = put_byte<G, 7>(out[7], hi);
}

// Member / branch masks of a thread's 32 symbols for every node.  The table gives a symbol's member byte and branch
// byte (bit v = node v); eight symbols' bytes are an 8x8 bit matrix whose transpose holds, in byte v, node v's bits of
// those eight symbols -- 24 instructions per matrix instead of a multiply-gather per node and four symbols.
template <int G>
__device__ __forceinline__ void wt_masks_group(const uint16_t *lut16, uint32_t w0, uint32_t w1, int n_internal,
                                               uint32_t (&m)[kWtSmallNodes], uint32_t (&b)[kWtSmallNodes])
{
    uint32_t M[2], B[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const uint32_t w = h ? w1 : w0;
        const uint32_t e0 = lut16[w & 0xff], e1 = lut16[(w >> 8) & 0xff], e2 = lut16[(w >> 16) & 0xff], e3 = lut16[w >> 24];
        const uint32_t lo = e0 | (e1 << 16), hi = e2 | (e3 << 16); // [mem0 br0 mem1 br1], [mem2 br2 mem3 br3]
        M[h] = __byte_perm(lo, hi, 0x6420);
        B[h] = __byte_perm(lo, hi, 0x7531);
    }
    transpose8x8(M[0], M[1]);
    transpose8x8(B[0], B[1]);
    wt_put_group<G>(M[0], M[1], n_internal, m);
    wt_put_group<G>(B[0], B[1], n_internal, b);
}

__device__ __forceinline__ void wt_masks_small(const uint16_t *lut16, const uint32_t (&w)[8], uint32_t valid, int n_internal,
                                               uint32_t (&m)[kWtSmallNodes], uint32_t (&b)[kWtSmallNodes])
{
#pragma unroll
    for (int v = 0; v < kWtSmallNodes; ++v) m[v] = b[v] = 0;
    wt_masks_group<0>(lut16, w[0], w[1], n_internal, m, b);
    wt_masks_group<1>(lut16, w[2], w[3], n_internal, m, b);
    wt_masks_group<2>(lut16, w[4], w[5], n_internal, m, b);
    wt_masks_group<3>(lut16, w[6], w[7], n_internal, m, b);
#pragma unroll
    for (int v = 0; v < kWtSmallNodes; ++v) {
        m[v] &= valid;
        b[v] &= valid;
    }
}

__global__ void __launch_bounds__(256)
wt_count_kernel(const uint8_t *__restrict__ seq, uint64_t n, const uint8_t *__restrict__ node_info, int n_internal,
                uint64_t ntiles, uint64_t *__restrict__ tile_count)
{
    extern __shared__ uint8_t s_info[];
    __shared__ uint32_t s_sum[8];
    __shared__ uint16_t s_lut16[256];
    __shared__ uint32_t s_part[kWtSmallNodes][8];
    const uint64_t tile = blockIdx.x;
    const uint64_t p0 = tile * kWtTile + (uint64_t)threadIdx.x * 32;
    uint32_t w[8];
    wt_load32(seq, n, p0, w);
    const uint32_t valid = wt_valid_mask(n, p0);
    if (n_internal <= kWtSmallNodes) {
        wt_small_table(node_info, n_internal, s_lut16);
        __syncthreads();
        uint32_t m[kWtSmallNodes], b[kWtSmallNodes];
        wt_masks_small(s_lut16, w, valid, n_internal, m, b);
#pragma unroll
        for (int v = 0; v < kWtSmallNodes; ++v) {
            if (v < n_internal) {
                const uint32_t c = warp_sum((uint32_t)__popc(m[v]));
                if ((threadIdx.x & 31) == 0) s_part[v][threadIdx.x >> 5] = c;
            }
        }
        __syncthreads();
        if (threadIdx.x < n_internal) {
            uint32_t t = 0;
            for (int k = 0; k < 8; ++k) t += s_part[threadIdx.x][k];
            tile_count[(uint64_t)threadIdx.x * ntiles + tile] = t;
        }
        return;
    }
    const bool staged = n_internal <= kWtInfoSmemNodes;
    if (staged) {
        for (int i = threadIdx.x; i < n_internal * 256; i += 256) s_info[i] = node_info[i];
        __syncthreads();
    }
    const uint8_t *info = staged ? s_info : node_info;
    for (int v = 0; v < n_internal; ++v) {
        uint32_t m, b;
        wt_masks(info + v * 256, w, valid, m, b);
        uint32_t c = warp_sum((uint32_t)__popc(m));
        if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t t = 0;
            for (int k = 0; k < 8; ++k) t += s_sum[k];
            tile_count[(uint64_t)v * ntiles + tile] = t;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) wt_scan_kernel(uint64_t *__restrict__ tile_count, uint64_t ntiles)
{
    __shared__ uint64_t scratch[33];
    uint64_t *row = tile_count + (uint64_t)blockIdx.x * ntiles;
    uint64_t carry = 0;
    for (uint64_t base = 0; base < ntiles; base += 1024) {
        const uint64_t i = base + threadIdx.x;
        const uint64_t v = i < ntiles ? row[i] : 0;
        uint64_t total;
        const uint64_t e = block_excl_sum(v, scratch, &total);
        if (i < ntiles) row[i] = carry + e;
        carry += total;
    }
}

// the bits of one node contributed by one thread: software pext of the branch bits over the member mask, OR-ed
// into the node's bit array at the thread's global bit offset
__device__ __forceinline__ void wt_emit(uint32_t m, uint32_t b, uint32_t c, uint64_t local, int v, const uint32_t (&w)[8],
                                        uint64_t *const *__restrict__ node_data, uint8_t *__restrict__ node_ch,
                                        const uint64_t *__restrict__ bit_base)
{
    uint64_t bits = b; // all 32 symbols are members (always so at the root): nothing to compress
    if (m != 0xffffffffu) {
        bits = 0;
        uint32_t mm = m;
        int out = 0;
        while (mm) {
            const int j = __ffs(mm) - 1;
            bits |= (uint64_t)((b >> j) & 1u) << out;
            ++out;
            mm &= mm - 1;
        }
    }
    const uint64_t o = local + (bit_base ? bit_base[v] : 0ull); // bit offset in the node's array
    unsigned long long *d = reinterpret_cast<unsigned long long *>(node_data[v]);
    const int sh = (int)(o & 63);
    if (bits << sh) atomicOr(d + (o >> 6), (unsigned long long)(bits << sh));
    if (sh + (int)c > 64 && (bits >> (64 - sh))) atomicOr(d + (o >> 6) + 1, (unsigned long long)(bits >> (64 - sh)));
    if (local == 0) { // first symbol of the node's subsequence (HuffWT.cpp:8)
        const int j = __ffs(m) - 1;
        node_ch[v] = (uint8_t)((w[j >> 2] >> (8 * (j & 3))) & 0xff);
    }
}

__global__ void __launch_bounds__(256)
wt_fill_kernel(const uint8_t *__restrict__ seq, uint64_t n, const uint8_t *__restrict__ node_info, int n_internal,
               uint64_t ntiles, const uint64_t *__restrict__ tile_off, uint64_t *const *__restrict__ node_data,
               uint8_t *__restrict__ node_ch, const uint64_t *__restrict__ bit_base)
{
    extern __shared__ uint8_t s_info[];
    __shared__ uint32_t scratch[9];
    __shared__ uint16_t s_lut16[256];
    __shared__ uint32_t s_part[kWtSmallNodes][8];
    const uint64_t tile = blockIdx.x;
    const uint64_t p0 = tile * kWtTile + (uint64_t)threadIdx.x * 32;
    uint32_t w[8];
    wt_load32(seq, n, p0, w);
    const uint32_t valid = wt_valid_mask(n, p0);
    if (n_internal <= kWtSmallNodes) {
        wt_small_table(node_info, n_internal, s_lut16);
        __syncthreads();
        uint32_t m[kWtSmallNodes], b[kWtSmallNodes], incl[kWtSmallNodes];
        wt_masks_small(s_lut16, w, valid, n_internal, m, b);
        // exclusive prefix of every node's member count over the threads of the tile: one barrier for all nodes
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int v = 0; v < kWtSmallNodes; ++v) {
            if (v < n_internal) {
                incl[v] = warp_incl_sum((uint32_t)__popc(m[v]));
                if (lane == 31) s_part[v][warp] = incl[v];
            }
        }
        __syncthreads();
#pragma unroll
        for (int v = 0; v < kWtSmallNodes; ++v) {
            if (v < n_internal) {
                const uint32_t c = __popc(m[v]);
                if (c) {
                    uint32_t before = incl[v] - c;
                    for (int k = 0; k < warp; ++k) before += s_part[v][k];
                    wt_emit(m[v], b[v], c, tile_off[(uint64_t)v * ntiles + tile] + before, v, w, node_data, node_ch, bit_base);
                }
            }
        }
        return;
    }
    const bool staged = n_internal <= kWtInfoSmemNodes;
    if (staged) {
        for (int i = threadIdx.x; i < n_internal * 256; i += 256) s_info[i] = node_info[i];
        __syncthreads();
    }
    const uint8_t *info = staged ? s_info : node_info;
    for (int v = 0; v < n_internal; ++v) {
        uint32_t m, b;
        wt_masks(info + v * 256, w, valid, m, b);
        const uint32_t c = __popc(m);
        uint32_t total;
        const uint32_t e = block_excl_sum(c, scratch, &total);
        if (c) wt_emit(m, b, c, tile_off[(uint64_t)v * ntiles + tile] + e, v, w, node_data, node_ch, bit_base);
    }
}

// the bits of x selected by m, moved together to the low end (parallel suffix method, Hacker's Delight 7-4): 5 rounds
// of straight-line code whatever the mask
__device__ __forceinline__ uint32_t compress_bits(uint32_t x, uint32_t m)
{
    x &= m;
    uint32_t mk = ~m << 1;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        uint32_t mp = mk ^ (mk << 1);
        mp ^= mp << 2;
        mp ^= mp << 4;
        mp ^= mp << 8;
        mp ^= mp << 16;
        const uint32_t mv = mp & m;
        m = (m ^ mv) | (mv >> (1 << i));
        const uint32_t t = x & mv;
        x = (x ^ t) | (t >> (1 << i));
        mk &= ~mp;
    }
    return x;
}

// ---- one pass over the sequence for small trees (reads: 6 internal nodes) -----------------------------------
// wt_count + wt_scan + wt_fill read the sequence twice, build the member masks twice, and every thread ORs its
// bits into the node arrays with global atomics (two per node and thread).  For trees of at most 8 internal nodes
// one kernel does it all: a CTA takes the next tile (dynamic tile id), builds the masks once and publishes its member
// counts per node at once; the tile's bits of every node are assembled in shared memory from bit 0 (32-bit shared
// atomics), which needs no global offset; only then does the CTA obtain the bit offsets of its runs by decoupled
// look-back over the tiles in front (one warp per node, 32 predecessors per step) -- they published long ago, so
// the look-back hardly ever waits -- and the runs leave the SM as whole 64-bit words, shifted to their offset; only
// the first and the last word of a run, which it may share with its neighbours, are OR-ed into global memory.
constexpr int kWtRunWords = kWtTile / 64 + 2; // 64-bit words a tile's run of one node can touch

// NI: the number of internal nodes at compile time (reads: 6), 0 = run time.  With a run-time count the per-node loops
// are unrolled to 8 and predicated: a quarter of the issued instructions does nothing for a six-node tree.
template <int NI>
__global__ void __launch_bounds__(256)
wt_sweep_kernel(const uint8_t *__restrict__ seq, uint64_t n, const uint8_t *__restrict__ node_info, int n_internal_rt,
                volatile unsigned long long *status, uint32_t *counter, uint64_t *const *__restrict__ node_data,
                uint8_t *__restrict__ node_ch, const uint64_t *__restrict__ bit_base)
{
    const int n_internal = NI ? NI : n_internal_rt;
    __shared__ uint16_t s_lut16[256];
    __shared__ uint32_t s_part[kWtSmallNodes][8];
    __shared__ uint32_t s_total[kWtSmallNodes];
    __shared__ unsigned long long s_off[kWtSmallNodes]; // global bit offset of the tile's run in node v
    __shared__ uint32_t s_bits[kWtSmallNodes][2 * kWtRunWords]; // the tile's bits of node v, from bit 0
    __shared__ uint8_t s_first[kWtSmallNodes];          // first member symbol of node v in this tile
    __shared__ uint32_t s_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(counter, 1u);
    wt_small_table(node_info, n_internal, s_lut16);
    for (int i = tid; i < kWtSmallNodes * 2 * kWtRunWords; i += 256) (&s_bits[0][0])[i] = 0;
    __syncthreads();
    const uint64_t tile = s_tile;
    const uint64_t p0 = tile * kWtTile + (uint64_t)tid * 32;
    uint32_t w[8];
    wt_load32(seq, n, p0, w);
    const uint32_t valid = wt_valid_mask(n, p0);
    uint32_t m[kWtSmallNodes], b[kWtSmallNodes], incl[kWtSmallNodes];
    wt_masks_small(s_lut16, w, valid, n_internal, m, b);
#pragma unroll
    for (int v = 0; v < kWtSmallNodes; ++v) {
        if (v < n_internal) {
            incl[v] = warp_incl_sum((uint32_t)__popc(m[v]));
            if (lane == 31) s_part[v][warp] = incl[v];
        }
    }
    __syncthreads();
    // warp v: total of node v -- published at once, so that the tiles behind can go on; this tile's own look-back
    // comes last, after its bits are assembled, when the tiles in front have long published theirs
    uint32_t total = 0;
    volatile unsigned long long *st = status + (size_t)warp; // status[tile * 8 + node]
    if (warp < n_internal) {
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t pk = s_part[warp][k];
            if (k < lane) mine += pk;
            total += pk;
        }
        __syncwarp();
        if (lane < 8) s_part[warp][lane] = mine; // from here on: members of node `warp` in the warps in front of warp `lane`
        if (lane == 0) {
            st[tile * kWtSmallNodes] = (tile == 0 ? kSelFlagPrefix : kSelFlagAgg) | total;
            s_total[warp] = total;
        }
    }
    __syncthreads();
    // every thread: its bits of every node into the tile's run (bit 0 of the run buffer = the tile's first member)
#pragma unroll
    for (int v = 0; v < kWtSmallNodes; ++v) {
        if (v < n_internal) {
            const uint32_t c = __popc(m[v]);
            // many members somewhere in the warp (the two nodes under the root of a read collection): compress
            // without a loop, whose trip count would be the warp's maximum
            const bool dense = __any_sync(0xffffffffu, c > 12u && m[v] != 0xffffffffu);
            if (c) {
                const uint32_t before = incl[v] - c + s_part[v][warp];
                uint32_t bits = b[v]; // all 32 symbols are members (always so at the root): nothing to compress
                if (m[v] != 0xffffffffu) {
                    if (dense) {
                        bits = compress_bits(b[v], m[v]);
                    } else {
                        bits = 0;
                        uint32_t mm = m[v];
                        int out = 0;
                        while (mm) {
                            const int j = __ffs(mm) - 1;
                            bits |= ((b[v] >> j) & 1u) << out;
                            ++out;
                            mm &= mm - 1;
                        }
                    }
                }
                const int sh = (int)(before & 31);
                if (bits << sh) atomicOr(&s_bits[v][before >> 5], bits << sh);
                if (sh && (bits >> (32 - sh))) atomicOr(&s_bits[v][(before >> 5) + 1], bits >> (32 - sh));
                if (before == 0) { // the tile's first member of the node: the node's first symbol if the tile is its first (HuffWT.cpp:8)
                    const int j = __ffs(m[v]) - 1;
                    uint32_t word = w[0];
#pragma unroll
                    for (int q = 1; q < 8; ++q)
                        if ((j >> 2) == q) word = w[q];
                    s_first[v] = (uint8_t)((word >> (8 * (j & 3))) & 0xff);
                }
            }
        }
    }
    // warp v: look back for the bit offset of the tile's run in node v
    if (warp < n_internal) {
        unsigned long long excl = 0;
        if (tile != 0) {
            long long t = (long long)tile - 1;
            for (;;) {
                const long long idx = t - lane;
                unsigned long long x = 2ull << 62; // in front of the first tile: an empty prefix
                if (idx >= 0) x = st[idx * kWtSmallNodes];
                while (__any_sync(0xffffffffu, (x >> 62) == 0))
                    if ((x >> 62) == 0) x = st[idx * kWtSmallNodes];
                const uint32_t pm = __ballot_sync(0xffffffffu, (x >> 62) == 2);
                const int stop = pm ? __ffs(pm) - 1 : 32;
                unsigned long long val = lane <= stop ? (x & kSelValueMask) : 0ull;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) val += __shfl_xor_sync(0xffffffffu, val, d);
                excl += val;
                if (pm) break;
                t -= 32;
            }
            if (lane == 0) st[tile * kWtSmallNodes] = kSelFlagPrefix | (excl + total);
        }
        if (lane == 0) s_off[warp] = excl + (bit_base ? bit_base[warp] : 0ull);
    }
    __syncthreads();
    // the runs leave as whole 64-bit words, shifted to their bit offset; the first and the last word of a run may be
    // shared with the neighbouring tiles and are OR-ed in
    for (int v = 0; v < n_internal; ++v) {
        const uint32_t tot = s_total[v];
        if (!tot) continue;
        const uint64_t off = s_off[v];
        const int sh = (int)(off & 63);
        if (tid == 0 && off == (bit_base ? bit_base[v] : 0ull)) node_ch[v] = s_first[v];
        const uint32_t words = (uint32_t)((sh + tot + 63) >> 6);
        unsigned long long *d = reinterpret_cast<unsigned long long *>(node_data[v]) + (off >> 6);
        for (uint32_t i = tid; i < words; i += 256) {
            const unsigned long long cur = (unsigned long long)s_bits[v][2 * i] | ((unsigned long long)s_bits[v][2 * i + 1] << 32);
            unsigned long long x = cur << sh;
            if (sh && i) {
                const unsigned long long prv = (unsigned long long)s_bits[v][2 * i - 2] | ((unsigned long long)s_bits[v][2 * i - 1] << 32);
                x |= prv >> (64 - sh);
            }
            if (i == 0 || i + 1 == words) {
                if (x) atomicOr(d + i, x);
            } else {
                d[i] = x;
            }
        }
    }
}

// Pieces of node bit arrays built by different GPUs (each already shifted to its global bit offset modulo
// 64) are merged into the node arrays: interior words are plain copies, the first and last word of a piece
// may share their destination word with a neighbouring piece and are OR-ed in.
__global__ void __launch_bounds__(256) wt_merge_pieces_kernel(const uint64_t *__restrict__ src, const WtPiece *__restrict__ pieces)
{
    const WtPiece pc = pieces[blockIdx.y];
    const uint64_t *from = src + pc.src_word;
    unsigned long long *to = reinterpret_cast<unsigned long long *>(pc.dst);
    const uint64_t stride = (uint64_t)gridDim.x * 256;
    for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < pc.nwords; i += stride) {
        const uint64_t x = from[i];
        if (i == 0 || i + 1 == pc.nwords) {
            if (x) atomicOr(to + i, (unsigned long long)x);
        } else {
            to[i] = x;
        }
    }
}

// BitRank: popcount of every chunk of kRankChunk superblocks
__global__ void __launch_bounds__(256) rank_chunk_sum_kernel(const uint64_t *__restrict__ data, uint64_t integers,
                                                             uint64_t *__restrict__ chunk_sum)
{
    __shared__ uint64_t s[8];
    const uint64_t w0 = (uint64_t)blockIdx.x * kRankChunk * 4;
    uint64_t c = 0;
    for (int i = threadIdx.x; i < kRankChunk * 4; i += 256) {
        const uint64_t w = w0 + i;
        if (w < integers) c += __popcll(data[w]);
    }
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t t = 0;
        for (int k = 0; k < 8; ++k) t += s[k];
        chunk_sum[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) rank_chunk_scan_kernel(uint64_t *__restrict__ chunk_sum, uint64_t nchunks)
{
    __shared__ uint64_t scratch[33];
    uint64_t carry = 0;
    for (uint64_t base = 0; base < nchunks; base += 1024) {
        const uint64_t i = base + threadIdx.x;
        const uint64_t v = i < nchunks ? chunk_sum[i] : 0;
        uint64_t total;
        const uint64_t e = block_excl_sum(v, scratch, &total);
        if (i < nchunks) chunk_sum[i] = carry + e;
        carry += total;
    }
}

__global__ void __launch_bounds__(256)
rank_write_kernel(const uint64_t *__restrict__ data, uint64_t integers, uint64_t nbits,
                  const uint64_t *__restrict__ chunk_base, uint64_t *__restrict__ Rs, uint8_t *__restrict__ Rb,
                  uint64_t base)
{
    constexpr int SB_PER_THREAD = kRankChunk / 256; // 8
    __shared__ uint64_t scratch[9];
    const uint64_t nsb = nbits / 256, nb = nbits / 64;
    const uint64_t sb0 = (uint64_t)blockIdx.x * kRankChunk + (uint64_t)threadIdx.x * SB_PER_THREAD;
    uint32_t cnt[SB_PER_THREAD];
    uint64_t mine = 0;
#pragma unroll
    for (int q = 0; q < SB_PER_THREAD; ++q) {
        const uint64_t j = sb0 + q;
        uint32_t run = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const uint64_t k = 4 * j + t;
            if (k <= nb) Rb[k] = (uint8_t)run;
            if (k < integers) run += __popcll(data[k]);
        }
        cnt[q] = run;
        mine += run;
    }
    uint64_t total;
    uint64_t e = block_excl_sum(mine, scratch, &total) + chunk_base[blockIdx.x] + base;
#pragma unroll
    for (int q = 0; q < SB_PER_THREAD; ++q) {
        const uint64_t j = sb0 + q;
        if (j <= nsb) Rs[j] = e;
        e += cnt[q];
    }
}

int grid_for(uint64_t items, int per_cta, int max_waves = 8)
{
    uint64_t want = div_up(items ? items : 1, (uint64_t)per_cta);
    uint64_t cap = (uint64_t)kNumSMs * max_waves;
    return (int)(want < cap ? want : cap);
}

#define DISPATCH_BITS(bits, CALL)                                                                     \
    do {                                                                                              \
        if ((bits) == 3) { CALL(3); }                                                                 \
        else if ((bits) == 4) { CALL(4); }                                                            \
        else if ((bits) == 8) { CALL(8); }                                                            \
        else throw CudaError{cudaErrorInvalidValue, "unsupported bits per symbol", __FILE__, __LINE__}; \
    } while (0)

} // namespace

// ---------------------------------------------------------------------------
// launch wrappers
// ---------------------------------------------------------------------------
void launch_byte_hist(cudaStream_t st, const uint8_t *raw, uint64_t n, uint64_t *counts, uint32_t *launches)
{
    byte_hist_kernel<<<grid_for(n, 256 * 64), 256, 0, st>>>(raw, n, counts);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_doc_stats(cudaStream_t st, const uint8_t *raw, uint64_t n, ChunkStat *out, uint32_t *launches)
{
    if (n == 0) return;
    doc_stats_kernel<<<(unsigned)div_up(n, kStatChunk), 256, 0, st>>>(raw, n, out);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_pack(cudaStream_t st, int bits, const uint8_t *raw, uint64_t n, const uint8_t *code_map, uint64_t *packed,
                 uint64_t nwords, uint32_t *launches)
{
#define CALL(B) pack_kernel<B><<<grid_for(nwords, 256), 256, 0, st>>>(raw, n, code_map, packed, nwords)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

// The fast kernels classify by the top 12 key bits; they apply when the first key has at least 12 bits
// and at least TopBits::SYMS symbols (always, except under DSMFM_FIRST_KEY_BITS experiments).
static bool select_fast_ok(int bits, int first_syms, int top_bits)
{
    const int syms = bits == 8 ? 2 : 12 / bits;
    return top_bits == 12 && first_syms >= syms;
}

void launch_make_keys_hist(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n, uint64_t *keys, int first_syms,
                           bool carry_prev, uint64_t *ghist, uint32_t *launches, uint64_t word_begin, uint64_t word_end)
{
    const int key_bits = first_syms * bits;
    const int npass = (key_bits + 7) / 8;
    uint64_t nwords = div_up(n, 64 / bits);
    if (word_end && word_end < nwords) nwords = word_end;
    if (word_begin >= nwords) return;
    const int grid = grid_for(nwords - word_begin, kKeyTileThreads, 16);
#define CALL(B)                                                                                                       \
    do {                                                                                                              \
        if (npass == 6)                                                                                               \
            make_keys_hist_kernel<B, 6><<<grid, kKeyTileThreads, 0, st>>>(packed, n, word_begin, nwords, keys, key_bits, \
                                                                          carry_prev, npass, ghist);                  \
        else                                                                                                          \
            make_keys_hist_kernel<B, -1><<<grid, kKeyTileThreads, 0, st>>>(packed, n, word_begin, nwords, keys, key_bits, \
                                                                           carry_prev, npass, ghist);                 \
    } while (0)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_key_top_hist(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n, int first_syms, int top_bits,
                         unsigned long long *hist, uint32_t *launches)
{
    const int drop_bits = (64 / bits - first_syms) * bits;
    const int top_shift = first_syms * bits - top_bits;
    const uint64_t nwords = div_up(n, 64 / bits);
    if (select_fast_ok(bits, first_syms, top_bits)) {
#define CALL(B) key_top_hist_fast_kernel<B><<<grid_for(nwords, 256 * 4), 256, 0, st>>>(packed, n, nwords, hist)
        DISPATCH_BITS(bits, CALL);
#undef CALL
    } else {
#define CALL(B) key_top_hist_kernel<B><<<grid_for(n, 256 * 16), 256, 0, st>>>(packed, n, drop_bits, top_shift, hist)
        DISPATCH_BITS(bits, CALL);
#undef CALL
    }
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

uint64_t select_tiles(uint64_t nwords, int bits, int first_syms, int top_bits)
{
    if (select_fast_ok(bits, first_syms, top_bits)) return div_up(nwords, (uint64_t)kSweepSelWords * kSelSub);
    return div_up(nwords * (uint64_t)(64 / bits), kSelTile);
}

// top 12 key bits of a suffix from the raw (uncut) leading bits: the host mirror of top_bin()
static uint32_t host_top_bin(int bits, uint32_t raw)
{
    const int syms = bits == 8 ? 2 : 12 / bits, rawbits = syms * bits;
    uint32_t x = 0;
    for (int i = 0; i < syms; ++i) { // fields from the most significant on; everything after the first zero field is cut
        const uint32_t f = (raw >> (rawbits - bits * (i + 1))) & ((1u << bits) - 1u);
        if (!f) break;
        x |= f << (rawbits - bits * (i + 1));
    }
    return x >> (rawbits - 12);
}

void launch_select(cudaStream_t st, int bits, const uint64_t *packed, uint64_t nwords, int first_syms, int top_bits,
                   bool carry_prev, uint64_t key_lo, uint64_t key_hi, uint64_t *tile_scratch, uint32_t *counter,
                   uint64_t *keys, uint32_t *vals, int lo_bits, int hi_shift, const SelGeom &geom, uint32_t *lut_scratch,
                   uint32_t *launches)
{
    const int drop_bits = (64 / bits - first_syms) * bits;
    const int key_bits = first_syms * bits;
    const unsigned tiles = (unsigned)select_tiles(nwords, bits, first_syms, top_bits);
    if (select_fast_ok(bits, first_syms, top_bits) && carry_prev) {
        const int sh = key_bits - 12;
        const uint32_t bin_lo = (uint32_t)(key_lo >> sh), bin_hi = (uint32_t)(key_hi >> sh);
        const int rawbits = (bits == 8 ? 2 : 12 / bits) * bits;
        std::vector<uint32_t> lut((size_t)1 << (rawbits - 5), 0u);
        for (uint32_t raw = 0; raw < (1u << rawbits); ++raw) {
            const uint32_t bin = host_top_bin(bits, raw);
            if (bin >= bin_lo && bin < bin_hi) lut[raw >> 5] |= 1u << (raw & 31);
        }
        // (pageable source: the copy has left the vector when the call returns)
        DSM_CUDA(cudaMemcpyAsync(lut_scratch, lut.data(), lut.size() * 4, cudaMemcpyHostToDevice, st));
        DSM_CUDA(cudaMemsetAsync(tile_scratch, 0, (size_t)tiles * 8, st));
        DSM_CUDA(cudaMemsetAsync(counter, 0, 4, st));
#define CALL(B)                                                                                                        \
    select_sweep_kernel<B><<<tiles, kSweepSelThreads, 0, st>>>(                                                        \
        packed, nwords, key_bits, lut_scratch, geom, reinterpret_cast<volatile unsigned long long *>(tile_scratch),     \
        counter, keys, vals, lo_bits, hi_shift)
        DISPATCH_BITS(bits, CALL);
#undef CALL
        DSM_LAUNCH_CHECK();
        if (launches) ++*launches;
        return;
    }
    // generic path (first keys shorter than 12 bits: only under DSMFM_FIRST_KEY_BITS experiments, one block only)
    if (geom.world != 1)
        throw CudaError{cudaErrorInvalidValue, "key-range selection over several blocks needs a first key of >= 12 bits", __FILE__, __LINE__};
    const uint64_t n = geom.bytes[0];
#define CALL(B) select_count_kernel<B><<<tiles, 256, 0, st>>>(packed, n, drop_bits, key_lo, key_hi, tile_scratch)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    launch_wt_scan(st, tile_scratch, 1, tiles, launches);
#define CALL(B)                                                                                                   \
    select_write_kernel<B><<<tiles, 256, 0, st>>>(packed, n, drop_bits, key_bits, carry_prev, key_lo, key_hi,     \
                                                  tile_scratch, keys, vals, lo_bits, hi_shift)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 2;
}

void launch_heads(cudaStream_t st, int bits, const uint64_t *sorted_keys, uint64_t n, uint32_t *head,
                  uint64_t head_words, unsigned long long *remaining, int key_bits, const uint8_t *inv_map,
                  uint8_t *bwt, uint8_t *pos_hi, int hi_shift, uint32_t *diff, uint32_t *launches)
{
#define CALL(B)                                                                                                      \
    heads_kernel<B><<<grid_for(head_words, 8 * 16), 256, 0, st>>>(sorted_keys, n, head, head_words, remaining, key_bits, \
                                                                   inv_map, bwt, pos_hi, hi_shift, diff)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

uint32_t launch_refine(cudaStream_t st, int bits, const uint64_t *packed, uint32_t *sa, const uint32_t *head_cur,
                   uint32_t *head_next, uint64_t n, uint32_t depth, const uint32_t *win_list, uint32_t n_list,
                   uint32_t *big_heads, uint32_t big_cap, uint32_t *big_count, unsigned long long *remaining,
                   uint32_t *win_flag, uint32_t *win_next, uint32_t *win_next_count, uint8_t *bwt, uint8_t *sa_hi,
                   int lo_bits, bool full_order, const uint32_t *diff_bits, uint32_t *launches, bool big_groups)
{
    const unsigned grid = win_list ? n_list : (unsigned)div_up(n, kRefWindow);
    if (grid == 0) return 0;
    // groups of at least big_thr members are ranked by the whole warp around their dominant key
    // (DSMFM_REFINE_BIG=<members>; 0 or unset: every group by its own members)
    // -- the default when the refinement runs in place, i.e. when most suffixes sit in groups that have to be
    // sorted (high repetition: C5 refinement 118 -> 98 ms); on the dense arrays of a read collection with few
    // large groups the per-member path is the faster one (C3: 25.2 vs 26.6 ms).
    const char *big_str = std::getenv("DSMFM_REFINE_BIG"); // (read per launch: the tests switch it)
    const int big_env = big_str ? std::atoi(big_str) : -1;
    const int big_want = big_env >= 0 ? big_env : (big_groups ? kRwBigGroup : 0);
    const int big_thr = big_want >= 32 ? (big_want < kRwBigGroup ? kRwBigGroup : big_want) : kRwCap + 1;
    static DeviceOnce attr_once;
    attr_once.run([] {
#define SET2(B, W, O)                                                                                                 \
    DSM_CUDA(cudaFuncSetAttribute(refine_warps_kernel<B, W, O, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                  (int)sizeof(RwSmem<W>)));                                                         \
    DSM_CUDA(cudaFuncSetAttribute(refine_warps_kernel<B, W, O, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                  (int)sizeof(RwSmem<W>)))
#define SET(B) SET2(B, false, false); SET2(B, true, false); SET2(B, false, true); SET2(B, true, true)
        SET(3); SET(4); SET(8);
#undef SET
#undef SET2
    });
    uint32_t ran = 0; // the instantiation launched, set beside its launch
#define RW2(B, W, O, C)                                                                                           \
    (refine_warps_kernel<B, W, O, C><<<grid, kRefThreads, sizeof(RwSmem<W>), st>>>(                               \
         packed, sa, head_cur, head_next, n, depth, win_list, big_heads, big_cap, big_count, remaining, win_flag, \
         win_next, win_next_count, bwt, sa_hi, lo_bits, diff_bits, big_thr),                                     \
     ran = (uint32_t)B << kRwLaunchedBitsShift | (W ? kRwLaunchedWide : 0u) | (O ? kRwLaunchedOrder : 0u) |      \
           (C ? kRwLaunchedCoop : 0u))
#define RW(B, W, O)                                                                                               \
    do {                                                                                                          \
        if (big_thr <= kRwCap) RW2(B, W, O, true); else RW2(B, W, O, false);                                      \
    } while (0)
#define CALL(B)                                                                                                   \
    do {                                                                                                          \
        if (full_order || !bwt) {                                                                                 \
            if (sa_hi) RW(B, true, true); else RW(B, false, true);                                                \
        } else {                                                                                                  \
            if (sa_hi) RW(B, true, false); else RW(B, false, false);                                              \
        }                                                                                                         \
    } while (0)
    DISPATCH_BITS(bits, CALL);
#undef CALL
#undef RW
#undef RW2
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
    return ran;
}

uint64_t active_tiles(uint64_t head_words) { return div_up(head_words, kActTileWords); }

void launch_mark_active(cudaStream_t st, const uint32_t *head, const uint32_t *diff, uint64_t n, uint32_t *act,
                        uint64_t *tile_off, uint32_t *launches)
{
    const uint64_t nwords = div_up(n, 32);
    const unsigned tiles = (unsigned)active_tiles(nwords);
    mark_active_kernel<<<(unsigned)div_up(nwords, 256 * 4), 256, 0, st>>>(head, diff, nwords, act);
    count_active_kernel<<<tiles, 256, 0, st>>>(act, nwords, tile_off);
    scan_tiles_kernel<<<1, 1024, 0, st>>>(tile_off, tiles);
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 3;
}

void launch_compact_active(cudaStream_t st, const uint32_t *act, const uint32_t *head, uint64_t n, const uint64_t *tile_off,
                           const uint32_t *sa, const uint8_t *bwt, const uint8_t *sa_hi, uint64_t m_act, uint32_t *csa,
                           uint8_t *cbw, uint8_t *chi, uint32_t *corig, uint32_t *chead, uint64_t chead_words,
                           uint32_t *launches)
{
    const uint64_t nwords = div_up(n, 32);
    compact_active_kernel<<<(unsigned)active_tiles(nwords), 256, 0, st>>>(act, head, nwords, tile_off, sa, bwt, sa_hi, csa,
                                                                          cbw, chi, corig, chead);
    pad_heads_kernel<<<grid_for(chead_words - (m_act >> 5), 256), 256, 0, st>>>(chead, m_act, chead_words);
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 2;
}

void launch_scatter_bwt(cudaStream_t st, const uint32_t *corig, const uint8_t *cbw, uint64_t m_act, uint8_t *bwt,
                        uint32_t *launches)
{
    scatter_bwt_kernel<<<grid_for(m_act, 256 * 8), 256, 0, st>>>(corig, cbw, m_act, bwt);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_big_extent(cudaStream_t st, const uint32_t *head_cur, uint64_t n, const uint32_t *big_heads, uint32_t nbig,
                       uint32_t *big_len, uint32_t *launches)
{
    big_extent_kernel<<<(unsigned)div_up(nbig, 8), 256, 0, st>>>(head_cur, n, big_heads, nbig, big_len);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_big_gather(cudaStream_t st, int bits, const uint64_t *packed, const uint32_t *sa, uint32_t depth,
                       const uint32_t *big_heads, const uint64_t *big_off, uint32_t nbig, uint64_t total, uint32_t *bsa,
                       uint64_t *bkey, uint32_t *bgid, const uint8_t *sa_hi, uint8_t *bhi, int lo_bits,
                       uint32_t *launches)
{
#define CALL(B)                                                                                                    \
    big_gather_kernel<B><<<grid_for(total, 256 * 4), 256, 0, st>>>(packed, sa, depth, big_heads, big_off, nbig, total, \
                                                                   bsa, bkey, bgid, sa_hi, bhi, lo_bits)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_gather_u32_to_u64(cudaStream_t st, const uint32_t *src, const uint32_t *perm, uint64_t n, uint64_t *dst,
                              uint32_t *launches)
{
    gather_u32_to_u64_kernel<<<grid_for(n, 256 * 4), 256, 0, st>>>(src, perm, n, dst);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_big_scatter(cudaStream_t st, int bits, const uint32_t *perm, const uint32_t *bsa, const uint64_t *bkey,
                        const uint32_t *bgid, const uint32_t *big_heads, const uint64_t *big_off, uint64_t total,
                        uint32_t *sa, uint32_t *head_next, uint32_t *win_flag, uint32_t *win_next,
                        uint32_t *win_next_count, const uint64_t *packed, const uint8_t *inv_map, uint8_t *bwt,
                        const uint8_t *bhi, uint8_t *sa_hi, int lo_bits, uint32_t *launches)
{
#define CALL(B)                                                                                                   \
    big_scatter_kernel<B><<<grid_for(total, 256 * 4), 256, 0, st>>>(perm, bsa, bkey, bgid, big_heads, big_off, total, \
                                                                    sa, head_next, win_flag, win_next, win_next_count,      \
                                                                    packed, inv_map, bwt, bhi, sa_hi, lo_bits)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_widen_sa(cudaStream_t st, const uint32_t *lo, const uint8_t *hi, int lo_bits, uint64_t n, uint64_t *out,
                     uint32_t *launches)
{
    if (n == 0) return;
    widen_sa_kernel<<<grid_for(n, 256 * 4), 256, 0, st>>>(lo, hi, lo_bits, n, out);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_bwt(cudaStream_t st, int bits, const uint64_t *packed, const uint8_t *inv_map, const uint32_t *sa,
                uint64_t n, uint8_t *bwt, uint32_t *launches)
{
#define CALL(B) bwt_kernel<B><<<grid_for(n, 256 * 16), 256, 0, st>>>(packed, inv_map, sa, n, bwt)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

uint64_t term_tiles(uint64_t n) { return div_up(n, kTermTile); }

void launch_term_positions(cudaStream_t st, const uint8_t *raw, uint64_t n, uint64_t *tile_scratch, uint32_t *doc_end,
                           uint32_t *launches)
{
    const unsigned tiles = (unsigned)term_tiles(n);
    term_count_kernel<<<tiles, 256, 0, st>>>(raw, n, tile_scratch);
    DSM_LAUNCH_CHECK();
    launch_wt_scan(st, tile_scratch, 1, tiles, launches);
    term_write_kernel<<<tiles, 256, 0, st>>>(raw, n, tile_scratch, doc_end);
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 2;
}

void launch_sa_mark(cudaStream_t st, const uint32_t *doc_end, uint32_t ndocs, uint32_t rate, uint32_t *mark,
                    uint32_t *launches)
{
    sa_mark_kernel<<<(unsigned)div_up(ndocs, 256), 256, 0, st>>>(doc_end, ndocs, rate, mark);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_sa_rank_bits(cudaStream_t st, const uint32_t *sa, const uint8_t *bwt, const uint32_t *mark, uint64_t n,
                         uint32_t *out, uint64_t out_words, uint32_t *launches)
{
    sa_rank_bits_kernel<<<grid_for(out_words, 8 * 4), 256, 0, st>>>(sa, bwt, mark, n, out, out_words);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_sa_emit(cudaStream_t st, const uint32_t *sa, const uint64_t *bits, const uint64_t *Rs, const uint8_t *Rb,
                    uint64_t n, const uint32_t *doc_end, uint32_t ndocs, uint32_t *out_doc, uint32_t *out_off,
                    uint32_t *launches)
{
    sa_emit_kernel<<<grid_for(n, 256 * 8), 256, 0, st>>>(sa, bits, Rs, Rb, n, doc_end, ndocs, out_doc, out_off);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_packed_term_positions(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n_text, const SelGeom &geom,
                                  uint64_t *tile_scratch, uint64_t *doc_end, uint32_t *launches)
{
    const unsigned tiles = (unsigned)term_tiles(n_text);
#define CALL(B) packed_term_count_kernel<B><<<tiles, 256, 0, st>>>(packed, n_text, geom, tile_scratch)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    launch_wt_scan(st, tile_scratch, 1, tiles, launches);
#define CALL(B) packed_term_write_kernel<B><<<tiles, 256, 0, st>>>(packed, n_text, geom, tile_scratch, doc_end)
    DISPATCH_BITS(bits, CALL);
#undef CALL
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 2;
}

void launch_sa_mark64(cudaStream_t st, const uint64_t *doc_end, uint32_t ndocs, uint32_t rate, uint64_t slot_syms,
                      uint32_t *mark, uint32_t *launches)
{
    if (ndocs == 0) return;
    sa_mark64_kernel<<<(unsigned)div_up(ndocs, 256), 256, 0, st>>>(doc_end, ndocs, rate, slot_syms, mark);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_sa_slice_bits(cudaStream_t st, const uint32_t *sa, const uint8_t *hi, int lo_bits, const uint8_t *bwt,
                          const uint32_t *mark, uint64_t m, uint64_t *sampled, uint64_t sampled_base, uint64_t *ends,
                          unsigned long long *counts, uint32_t *launches)
{
    if (m == 0) return;
    sa_slice_bits_kernel<<<grid_for(div_up(m, 32), 8 * 4), 256, 0, st>>>(sa, hi, lo_bits, bwt, mark, m,
                                                                          reinterpret_cast<uint32_t *>(sampled), sampled_base,
                                                                          reinterpret_cast<uint32_t *>(ends), counts);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_sa_emit64(cudaStream_t st, const uint32_t *sa, const uint8_t *hi, int lo_bits, const uint64_t *bits,
                      const uint64_t *Rs, const uint8_t *Rb, uint64_t bits_base, uint64_t rank_sub, uint64_t m,
                      const uint64_t *doc_end, uint32_t ndocs, uint64_t slot_syms, uint64_t *doc_out, uint64_t doc_bit0,
                      unsigned doc_w, uint64_t *off_out, uint64_t off_bit0, unsigned off_w, uint32_t *launches)
{
    if (m == 0 || ndocs == 0) return;
    sa_emit64_kernel<<<grid_for(m, 256 * 8), 256, 0, st>>>(sa, hi, lo_bits, bits, Rs, Rb, bits_base, rank_sub, m, doc_end, ndocs,
                                                           slot_syms, doc_out, doc_bit0, doc_w, off_out, off_bit0, off_w);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_sa_lengths(cudaStream_t st, const uint64_t *doc_end, uint64_t first, uint64_t count, uint64_t slot_syms,
                       uint64_t *out, uint64_t bit0, unsigned w, uint32_t *launches)
{
    if (count == 0 || w == 0) return;
    sa_lengths_kernel<<<grid_for(count, 256 * 8), 256, 0, st>>>(doc_end, first, count, slot_syms, out, bit0, w);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

static size_t wt_info_smem(int n_internal) { return n_internal <= kWtInfoSmemNodes ? (size_t)n_internal * 256 : 0; }

void launch_wt_count(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                     uint64_t ntiles, uint64_t *tile_count, uint32_t *launches)
{
    wt_count_kernel<<<(unsigned)ntiles, 256, wt_info_smem(n_internal), st>>>(seq, n, node_info, n_internal, ntiles,
                                                                            tile_count);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_wt_scan(cudaStream_t st, uint64_t *tile_count, int n_internal, uint64_t ntiles, uint32_t *launches)
{
    wt_scan_kernel<<<n_internal, 1024, 0, st>>>(tile_count, ntiles);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_wt_fill(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                    uint64_t ntiles, const uint64_t *tile_off, uint64_t *const *node_data, uint8_t *node_ch,
                    const uint64_t *bit_base, uint32_t *launches)
{
    wt_fill_kernel<<<(unsigned)ntiles, 256, wt_info_smem(n_internal), st>>>(seq, n, node_info, n_internal, ntiles,
                                                                           tile_off, node_data, node_ch, bit_base);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

bool wt_sweep_ok(int n_internal) { return n_internal <= kWtSmallNodes; }
uint64_t wt_sweep_status_words(uint64_t ntiles) { return ntiles * kWtSmallNodes; }

void launch_wt_sweep(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                     uint64_t ntiles, uint64_t *status, uint32_t *counter, uint64_t *const *node_data, uint8_t *node_ch,
                     const uint64_t *bit_base, uint32_t *launches)
{
    DSM_CUDA(cudaMemsetAsync(status, 0, sizeof(uint64_t) * wt_sweep_status_words(ntiles), st));
    DSM_CUDA(cudaMemsetAsync(counter, 0, sizeof(uint32_t), st));
#define WT_SWEEP(NI)                                                                                              \
    wt_sweep_kernel<NI><<<(unsigned)ntiles, 256, 0, st>>>(seq, n, node_info, n_internal,                          \
                                                         reinterpret_cast<volatile unsigned long long *>(status), \
                                                         counter, node_data, node_ch, bit_base)
    if (n_internal == 6) WT_SWEEP(6); // seven symbols: reads over ACGTN with the separator and the terminator
    else if (n_internal == 5) WT_SWEEP(5);
    else if (n_internal == 4) WT_SWEEP(4);
    else WT_SWEEP(0);
#undef WT_SWEEP
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_wt_merge_pieces(cudaStream_t st, const uint64_t *src, const WtPiece *pieces, uint32_t npieces,
                            uint32_t *launches)
{
    if (npieces == 0) return;
    wt_merge_pieces_kernel<<<dim3(kNumSMs * 2, npieces), 256, 0, st>>>(src, pieces);
    DSM_LAUNCH_CHECK();
    if (launches) ++*launches;
}

void launch_bitrank(cudaStream_t st, const uint64_t *data, uint64_t nbits, uint64_t *Rs, uint8_t *Rb, uint64_t *scratch,
                    uint32_t *launches, uint64_t base)
{
    const uint64_t integers = nbits / 64 + 1;
    const uint64_t nsb = nbits / 256 + 1; // superblock entries 0..nbits/256
    const unsigned nchunks = (unsigned)div_up(nsb, kRankChunk);
    rank_chunk_sum_kernel<<<nchunks, 256, 0, st>>>(data, integers, scratch);
    DSM_LAUNCH_CHECK();
    rank_chunk_scan_kernel<<<1, 1024, 0, st>>>(scratch, nchunks);
    DSM_LAUNCH_CHECK();
    rank_write_kernel<<<nchunks, 256, 0, st>>>(data, integers, nbits, scratch, Rs, Rb, base);
    DSM_LAUNCH_CHECK();
    if (launches) *launches += 3;
}

} // namespace dsmfm
