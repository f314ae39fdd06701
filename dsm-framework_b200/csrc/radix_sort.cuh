// radix_sort.cuh -- stable LSD radix sort of (u64 key, u32 value) pairs for sm_100a.
//
// One-sweep design: a single histogram kernel counts every digit of every pass
// up front; each pass is then ONE kernel in which a CTA ranks its tile in
// shared memory (warp ballot multi-split, per-warp digit counters), obtains the
// global offset of each of its 256 digit runs by decoupled look-back over the
// tiles before it, and writes keys and values out from a shared-memory staging
// buffer so that every digit run leaves the SM as one coalesced burst.
//
// This replaces the std::sort calls of the reference's suffix sorter
// (incbwt/misc/utils.cpp:212-221 initialSort, 236-262 prefixDoubling).
#pragma once
#include "common.cuh"

namespace dsmfm {

constexpr int kRadixBits = 8;
constexpr int kRadix = 1 << kRadixBits;
constexpr int kMaxPasses = 8;

// Tile of the one-sweep kernel: 4096 pairs, 256 threads x 16 pairs.
constexpr int kSweepTile = 4096;
constexpr int kSweepThreads = 256;
constexpr int kSweepItems = kSweepTile / kSweepThreads;
constexpr int kSweepCtasPerSm = 4;
// A launch handles at most this many pairs so that tile prefixes fit the
// 30-bit payload of a status word; longer inputs run as several portions.
constexpr uint64_t kSweepPortion = (uint64_t)kSweepTile * 131072; // 2^29

struct RadixWorkspace {
    uint64_t *hist = nullptr;     // [kMaxPasses][256] digit counts, then exclusive bases
    uint64_t *carry = nullptr;    // [2][256] per-portion running bases
    uint32_t *status = nullptr;   // [tiles per portion][256] look-back words
    uint32_t *counter = nullptr;  // dynamic tile id
    uint64_t status_tiles = 0;
    size_t bytes = 0;

    void allocate(uint64_t max_n);
    void release();
};

// How keys enter the first pass of a sort.
struct KeysFromArray {
    const uint64_t *keys;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const { return keys[i]; }
};

// Sorts n pairs on key bits [begin_bit, end_bit).  Input in (keys_a, vals_a);
// the buffers ping-pong every pass.  Returns the number of passes run: an odd
// count leaves the result in (keys_b, vals_b).  With iota_first the values of
// the first pass are the element indices 0..n-1 and vals_a is only written
// (it must still be a valid buffer: it is the destination of odd passes).
// `launches` (optional) is incremented per kernel launched.  ev_begin/ev_end
// (optional) are recorded around the one-sweep passes (histogram excluded).
// hist_ready: ws.hist[pass][256] already holds the digit counts of the keys (whoever produced the keys
// counted them on the way), so the histogram pass over the key array is skipped.
// keys_a and keys_b must be 16-byte aligned: every whole tile's keys arrive by one bulk copy.
int radix_sort_pairs(cudaStream_t stream, RadixWorkspace &ws, uint64_t *keys_a, uint32_t *vals_a, uint64_t *keys_b,
                     uint32_t *vals_b, uint64_t n, int begin_bit, int end_bit, bool iota_first,
                     uint32_t *launches, cudaEvent_t ev_begin = nullptr, cudaEvent_t ev_end = nullptr,
                     bool hist_ready = false);

} // namespace dsmfm
