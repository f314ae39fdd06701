// api.cu -- the C ABI of include/dsmfm.h: host-side orchestration of the
// sm_100a build kernels.  No CPU fallback: every computation on the data path
// (histogram, packing, suffix sorting, BWT, wavelet tree, rank directories)
// runs in the kernels of kernels.cu / radix_sort.cu; the host only builds the
// <=256-entry Huffman code table and the tree shape, and writes files.
#include "../../include/dsmfm.h"
#include "kernels.cuh"
#include <thread>
#include "fasta.cuh"
#include "radix_sort.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <fcntl.h>
#include <unistd.h>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <queue>
#include <string>
#include <vector>

using namespace dsmfm;

namespace {

thread_local std::string g_create_error;

// ---------------------------------------------------------------------------
// Memory: device buffers come from the device's stream-ordered pool
// (cudaMallocAsync) whose release threshold is raised so that a second build
// reuses the first one's memory instead of paying for 50 GB of cudaMalloc /
// cudaFree; pinned host buffers (section copies, append staging) are cached in
// a small process-wide pool for the same reason.  dsmfm_release_cached() gives
// both back.
// ---------------------------------------------------------------------------
double now_ms()
{
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}
thread_local double g_alloc_ms = 0.0;
std::atomic<unsigned long long> g_guard_violations{0};

// DSMFM_TRACE=1: wall-clock milestones of a process on stderr (cold-start costs -- context creation, first
// device allocations, pinned buffers -- are invisible to the CUDA-event timers in dsmfm_stats)
void trace(const char *what)
{
    static const bool on = std::getenv("DSMFM_TRACE") != nullptr;
    if (!on) return;
    static const double t0 = now_ms();
    static double last = t0;
    const double t = now_ms();
    std::fprintf(stderr, "[dsmfm %9.1f ms +%8.1f] %s\n", t - t0, t - last, what);
    last = t;
}

// Large device blocks (>= 32 MB) are kept in a process-wide cache keyed by their exact size: a build of the same
// shape finds every one of its buffers again without a driver call.  (The stream-ordered pool alone is not
// enough: when the sizes free at the moment do not match a request it carves up or remaps a larger block, and
// an 8 GB request then takes anything from 5 to 800 ms -- measured in the multi-GPU bench.)  A block is handed
// out again only after an event recorded at its release, so different streams may share the cache.  Smaller
// allocations stay in the stream-ordered pool.
struct BlockCache {
    static constexpr size_t kMinBytes = (size_t)32 << 20;
    struct Blk { void *p; size_t bytes; int dev; cudaEvent_t ready; };
    std::mutex mu;
    std::vector<Blk> free_;
    std::vector<Blk> live_; // blocks handed out (ready unused)
    size_t free_bytes = 0;

    void drop(size_t i)
    {
        Blk b = free_[i];
        free_.erase(free_.begin() + i);
        free_bytes -= b.bytes;
        int cur = 0;
        cudaGetDevice(&cur);
        if (cur != b.dev) cudaSetDevice(b.dev);
        cudaEventSynchronize(b.ready);
        cudaEventDestroy(b.ready);
        cudaFree(b.p);
        if (cur != b.dev) cudaSetDevice(cur);
    }
    void *get(size_t bytes, cudaStream_t st)
    {
        int dev = 0;
        DSM_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> g(mu);
        for (size_t i = free_.size(); i-- > 0;) {
            if (free_[i].dev != dev || free_[i].bytes != bytes) continue;
            Blk b = free_[i];
            free_.erase(free_.begin() + i);
            free_bytes -= b.bytes;
            DSM_CUDA(cudaStreamWaitEvent(st, b.ready, 0));
            cudaEventDestroy(b.ready);
            b.ready = nullptr;
            live_.push_back(b);
            return b.p;
        }
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaErrorMemoryAllocation) { // give back what is cached and try once more
            cudaGetLastError();
            while (!free_.empty()) drop(free_.size() - 1);
            e = cudaMalloc(&p, bytes);
        }
        if (e != cudaSuccess) throw CudaError{e, "cudaMalloc (device block cache)", __FILE__, __LINE__};
        live_.push_back(Blk{p, bytes, dev, nullptr});
        return p;
    }
    // true if p was one of ours
    bool put(void *p, cudaStream_t st)
    {
        std::lock_guard<std::mutex> g(mu);
        for (size_t i = 0; i < live_.size(); ++i) {
            if (live_[i].p != p) continue;
            Blk b = live_[i];
            live_.erase(live_.begin() + i);
            if (cudaEventCreateWithFlags(&b.ready, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventRecord(b.ready, st) != cudaSuccess) {
                cudaStreamSynchronize(st);
                cudaFree(b.p);
                return true;
            }
            free_.push_back(b);
            free_bytes += b.bytes;
            // blocks of shapes that do not come back must not pile up next to other users of the device (the caller's
            // own cudaMalloc, torch's allocator): at most 128 GB idle (a 16 Gbp 8-GPU build holds 77 GB), oldest go first.  (No driver query here: on a
            // box where other processes allocate, cudaMemGetInfo stalled this path for up to 200 ms.)
            while (free_bytes > ((size_t)128 << 30) && free_.size() > 1) drop(0);
            return true;
        }
        return false;
    }
    void trim(int dev)
    {
        std::lock_guard<std::mutex> g(mu);
        for (size_t i = free_.size(); i-- > 0;)
            if (dev < 0 || free_[i].dev == dev) drop(i);
    }
};
BlockCache g_blocks;

void *dev_alloc(size_t bytes, cudaStream_t st)
{
    void *p = nullptr;
    const double t0 = now_ms();
    if (bytes >= BlockCache::kMinBytes)
        p = g_blocks.get(bytes, st);
    else
        DSM_CUDA(cudaMallocAsync(&p, bytes ? bytes : 1, st));
    const double dt = now_ms() - t0;
    g_alloc_ms += dt;
    static const bool loud = std::getenv("DSMFM_TRACE_ALLOC") != nullptr;
    if (loud && dt > 1.0) std::fprintf(stderr, "[dsmfm alloc] %zu bytes took %.1f ms\n", bytes, dt);
    return p;
}
void dev_free(void *p, cudaStream_t st)
{
    if (!p) return;
    if (!g_blocks.put(p, st)) cudaFreeAsync(p, st);
}

struct PinnedPool {
    struct Buf { void *p; size_t bytes; bool busy; };
    std::mutex mu;
    std::vector<Buf> bufs;
    void *get(size_t bytes)
    {
        std::lock_guard<std::mutex> g(mu);
        int best = -1;
        for (size_t i = 0; i < bufs.size(); ++i)
            if (!bufs[i].busy && bufs[i].bytes >= bytes && (best < 0 || bufs[i].bytes < bufs[best].bytes)) best = (int)i;
        if (best >= 0 && bufs[best].bytes <= 2 * bytes + (1u << 20)) {
            bufs[best].busy = true;
            return bufs[best].p;
        }
        void *p = nullptr;
        DSM_CUDA(cudaMallocHost(&p, bytes ? bytes : 1));
        bufs.push_back(Buf{p, bytes, true});
        return p;
    }
    void put(void *p)
    {
        if (!p) return;
        std::lock_guard<std::mutex> g(mu);
        for (auto &b : bufs)
            if (b.p == p) b.busy = false;
    }
    void trim()
    {
        std::lock_guard<std::mutex> g(mu);
        for (size_t i = 0; i < bufs.size();) {
            if (!bufs[i].busy) {
                cudaFreeHost(bufs[i].p);
                bufs.erase(bufs.begin() + i);
            } else
                ++i;
        }
    }
};
PinnedPool g_pinned;

// Scratch of the FASTA front end: one device buffer per device that only grows and is shared by all builders
// of the process (a call holds the lock and ends with a stream synchronize, so the buffer is idle in between).
// The stream-ordered pool is fast when the sizes of a build repeat; the front end's sizes follow the input
// file, and carving them out of pooled blocks of other sizes stalled for 100+ ms per call.
struct ScratchArena {
    static constexpr int kMaxDev = 64;
    std::mutex mu;
    void *ptr[kMaxDev] = {};
    size_t cap[kMaxDev] = {};
    size_t hint[kMaxDev] = {}; // what the last call on the device would have liked to find
    void *reserve(int dev, size_t bytes)
    {
        if (dev < 0 || dev >= kMaxDev) throw CudaError{cudaErrorInvalidDevice, "scratch arena", __FILE__, __LINE__};
        if (cap[dev] >= bytes) return ptr[dev];
        if (ptr[dev]) cudaFree(ptr[dev]);
        ptr[dev] = nullptr;
        cap[dev] = 0;
        const size_t want = bytes + bytes / 8;
        const double t0 = now_ms();
        DSM_CUDA(cudaMalloc(&ptr[dev], want));
        g_alloc_ms += now_ms() - t0;
        cap[dev] = want;
        return ptr[dev];
    }
    void trim(int dev)
    {
        std::lock_guard<std::mutex> g(mu);
        for (int d = 0; d < kMaxDev; ++d) {
            if ((dev >= 0 && d != dev) || !ptr[d]) continue;
            cudaSetDevice(d);
            cudaFree(ptr[d]);
            ptr[d] = nullptr;
            cap[d] = hint[d] = 0;
        }
    }
};
ScratchArena g_fasta_arena;

// ---------------------------------------------------------------------------
// Huffman code table -- node::makecodetable / maketable, HuffWT.cpp:133-184.
// Same container (std::priority_queue over std::vector with std::greater),
// same push order (ascending byte value, counts > 0), same weight-only
// comparison, so libstdc++'s heap resolves ties exactly as in the reference.
// ---------------------------------------------------------------------------
struct HuffNode {
    uint64_t weight;
    int id; // index into the tree arrays
    bool operator>(const HuffNode &o) const { return weight > o.weight; }
};

struct HuffTree {
    std::vector<int> child0, child1, value;
};

void huff_assign(const HuffTree &t, int node, uint32_t code, uint32_t bits, dsmfm_code *tab, uint32_t *maxbits)
{
    if (t.child0[node] >= 0) {
        huff_assign(t, t.child0[node], code, bits + 1, tab, maxbits);
        huff_assign(t, t.child1[node], bits < 32 ? (code | (1u << bits)) : code, bits + 1, tab, maxbits);
    } else {
        tab[t.value[node]].code = code;
        tab[t.value[node]].bits = bits;
        if (bits > *maxbits) *maxbits = bits;
    }
}

uint32_t build_codetable(const uint64_t counts[256], dsmfm_code tab[256])
{
    HuffTree t;
    std::priority_queue<HuffNode, std::vector<HuffNode>, std::greater<HuffNode>> q;
    for (int i = 0; i < 256; ++i) {
        tab[i].count = counts[i];
        tab[i].bits = 0;
        tab[i].code = 0;
    }
    for (int i = 0; i < 256; ++i) {
        if (!counts[i]) continue;
        t.child0.push_back(-1);
        t.child1.push_back(-1);
        t.value.push_back(i);
        q.push(HuffNode{counts[i], (int)t.value.size() - 1});
    }
    if (q.empty()) return 0;
    while (q.size() > 1) {
        HuffNode c0 = q.top();
        q.pop();
        HuffNode c1 = q.top();
        q.pop();
        t.child0.push_back(c0.id);
        t.child1.push_back(c1.id);
        t.value.push_back(0);
        q.push(HuffNode{c0.weight + c1.weight, (int)t.value.size() - 1});
    }
    uint32_t maxbits = 0;
    huff_assign(t, q.top().id, 0u, 0u, tab, &maxbits);
    return maxbits;
}

// ---------------------------------------------------------------------------
// Wavelet tree shape from the code table, in the pre-order HuffWT::save uses
// (HuffWT.cpp:73-86): a node at `level` holding the symbols whose code starts
// with `prefix`; leaf iff a single symbol whose code ends here (HuffWT.cpp:35-40).
// ---------------------------------------------------------------------------
struct WtShape {
    std::vector<dsmfm_node> nodes;       // pre-order; pointers filled after the device pass
    std::vector<int> internal_of_node;   // node -> internal index or -1
    std::vector<uint8_t> info;           // [n_internal][256] membership/branch table for the kernels
    int n_internal = 0;
};

void shape_rec(const dsmfm_code *tab, uint32_t prefix, uint32_t level, WtShape &s)
{
    int members = 0, only = -1;
    uint64_t total = 0;
    const uint32_t pmask = level >= 32 ? 0xffffffffu : ((1u << level) - 1u);
    for (int c = 0; c < 256; ++c) {
        if (!tab[c].count || tab[c].bits < level || (tab[c].code & pmask) != prefix) continue;
        ++members;
        only = c;
        total += tab[c].count;
    }
    dsmfm_node nd;
    std::memset(&nd, 0, sizeof nd);
    if (members == 1 && tab[only].bits == level) {
        nd.leaf = 1;
        nd.ch = (uint8_t)only; // a leaf's subsequence is one repeated symbol, so s[0] is that symbol
        s.nodes.push_back(nd);
        s.internal_of_node.push_back(-1);
        return;
    }
    nd.leaf = 0;
    nd.nbits = total;
    nd.integers = total / 64 + 1; // == ceil((n+1)/64), BitRank.cpp:97-101
    const int v = s.n_internal++;
    s.info.resize((size_t)s.n_internal * 256, 0);
    for (int c = 0; c < 256; ++c) {
        if (!tab[c].count || tab[c].bits < level || (tab[c].code & pmask) != prefix) continue;
        s.info[(size_t)v * 256 + c] = (uint8_t)(1u | (((tab[c].code >> level) & 1u) << 1));
    }
    s.nodes.push_back(nd);
    s.internal_of_node.push_back(v);
    shape_rec(tab, prefix, level + 1, s);
    shape_rec(tab, prefix | (1u << level), level + 1, s);
}

size_t align8(size_t x) { return (x + 7) & ~(size_t)7; }

// Device-side wavelet tree + BitRank build for a byte sequence already in HBM.
struct WaveletResult {
    WtShape shape;
    uint8_t *d_sections = nullptr; // [data | Rs | Rb] per internal node, 8-byte aligned pieces
    size_t section_bytes = 0;
    std::vector<size_t> off_data, off_rs, off_rb; // per internal node
    uint8_t *d_ch = nullptr;                      // per internal node
    // host copies (pinned), filled by fetch()
    uint8_t *h_sections = nullptr;
    std::vector<uint8_t> h_ch;

    void release(cudaStream_t st = nullptr)
    {
        dev_free(d_sections, st);
        dev_free(d_ch, st);
        g_pinned.put(h_sections);
        d_sections = d_ch = h_sections = nullptr;
    }
};

// shape of the tree and layout of the sections for a code table
void wavelet_prepare(const dsmfm_code *tab, WaveletResult &r)
{
    r.shape = WtShape();
    shape_rec(tab, 0u, 0u, r.shape);
    const int m = r.shape.n_internal;
    if (m > kWtMaxNodes) throw CudaError{cudaErrorInvalidValue, "too many wavelet tree nodes", __FILE__, __LINE__};
    r.off_data.assign(m, 0);
    r.off_rs.assign(m, 0);
    r.off_rb.assign(m, 0);
    size_t off = 0;
    for (size_t i = 0; i < r.shape.nodes.size(); ++i) {
        const int v = r.shape.internal_of_node[i];
        if (v < 0) continue;
        const dsmfm_node &nd = r.shape.nodes[i];
        r.off_data[v] = off;
        off += nd.integers * 8;
        r.off_rs[v] = off;
        off += (nd.nbits / 256 + 1) * 8;
        r.off_rb[v] = off;
        off += align8(nd.nbits / 64 + 1);
    }
    r.section_bytes = off;
}

void wavelet_alloc(cudaStream_t st, WaveletResult &r)
{
    const int m = r.shape.n_internal;
    r.d_sections = static_cast<uint8_t *>(dev_alloc(r.section_bytes, st));
    r.d_ch = static_cast<uint8_t *>(dev_alloc((size_t)(m ? m : 1), st));
    DSM_CUDA(cudaMemsetAsync(r.d_sections, 0, r.section_bytes, st));
    DSM_CUDA(cudaMemsetAsync(r.d_ch, 0, (size_t)(m ? m : 1), st));
}

// Bits of every internal node for the byte sequence d_seq: node v's bits go to ptrs[v] (device pointers,
// zero-initialised arrays) starting at bit bit_base[v] (empty = 0); d_ch[v] = first member symbol.
// Synchronises the stream.  Returns the scratch bytes it used.
size_t wavelet_fill_bits(cudaStream_t st, const uint8_t *d_seq, uint64_t n, const WtShape &shape,
                         const std::vector<uint64_t *> &ptrs, const std::vector<uint64_t> &bit_base, uint8_t *d_ch,
                         uint32_t *launches)
{
    const int m = shape.n_internal;
    if (m == 0 || n == 0) return 0;
    const uint64_t ntiles = div_up(n, kWtTile);
    const char *sweep_env = std::getenv("DSMFM_WT_SWEEP"); // 0: count / scan / fill for small trees too (read per call: the tests switch it)
    const bool sweep = wt_sweep_ok(m) && !(sweep_env && std::atoi(sweep_env) == 0); // one pass (small trees) or count / scan / fill
    const size_t tile_bytes = sizeof(uint64_t) * (sweep ? wt_sweep_status_words(ntiles) + 1 : (size_t)m * ntiles);
    uint8_t *d_info = static_cast<uint8_t *>(dev_alloc((size_t)m * 256, st));
    uint64_t *d_tile = static_cast<uint64_t *>(dev_alloc(tile_bytes, st));
    uint64_t **d_ptrs = static_cast<uint64_t **>(dev_alloc(sizeof(uint64_t *) * m, st));
    uint64_t *d_base = bit_base.empty() ? nullptr : static_cast<uint64_t *>(dev_alloc(sizeof(uint64_t) * m, st));
    try {
        DSM_CUDA(cudaMemcpyAsync(d_info, shape.info.data(), (size_t)m * 256, cudaMemcpyHostToDevice, st));
        DSM_CUDA(cudaMemcpyAsync(d_ptrs, ptrs.data(), sizeof(uint64_t *) * m, cudaMemcpyHostToDevice, st));
        if (d_base) DSM_CUDA(cudaMemcpyAsync(d_base, bit_base.data(), sizeof(uint64_t) * m, cudaMemcpyHostToDevice, st));
        if (sweep) {
            launch_wt_sweep(st, d_seq, n, d_info, m, ntiles, d_tile,
                            reinterpret_cast<uint32_t *>(d_tile + wt_sweep_status_words(ntiles)), d_ptrs, d_ch, d_base, launches);
        } else {
            launch_wt_count(st, d_seq, n, d_info, m, ntiles, d_tile, launches);
            launch_wt_scan(st, d_tile, m, ntiles, launches);
            launch_wt_fill(st, d_seq, n, d_info, m, ntiles, d_tile, d_ptrs, d_ch, d_base, launches);
        }
        DSM_CUDA(cudaStreamSynchronize(st)); // the host vectors are consumed
    } catch (...) {
        dev_free(d_info, st); dev_free(d_tile, st); dev_free(d_ptrs, st); dev_free(d_base, st);
        throw;
    }
    dev_free(d_info, st);
    dev_free(d_tile, st);
    dev_free(d_ptrs, st);
    dev_free(d_base, st);
    return (size_t)m * 256 + tile_bytes + sizeof(uint64_t *) * m;
}

// BitRank directories of every internal node (data already in r.d_sections)
void wavelet_ranks(cudaStream_t st, WaveletResult &r, uint32_t *launches)
{
    uint64_t max_sb = 0;
    for (size_t i = 0; i < r.shape.nodes.size(); ++i)
        if (r.shape.internal_of_node[i] >= 0) max_sb = std::max<uint64_t>(max_sb, r.shape.nodes[i].nbits / 256 + 1);
    if (!max_sb) return;
    uint64_t *d_scratch = static_cast<uint64_t *>(dev_alloc(sizeof(uint64_t) * (div_up(max_sb, kRankChunk) + 1), st));
    try {
        for (size_t i = 0; i < r.shape.nodes.size(); ++i) {
            const int v = r.shape.internal_of_node[i];
            if (v < 0) continue;
            launch_bitrank(st, reinterpret_cast<uint64_t *>(r.d_sections + r.off_data[v]), r.shape.nodes[i].nbits,
                           reinterpret_cast<uint64_t *>(r.d_sections + r.off_rs[v]), r.d_sections + r.off_rb[v],
                           d_scratch, launches);
        }
    } catch (...) {
        dev_free(d_scratch, st);
        throw;
    }
    dev_free(d_scratch, st);
}

void wavelet_build_device(cudaStream_t st, const uint8_t *d_seq, uint64_t n, const dsmfm_code *tab, WaveletResult &r,
                          uint32_t *launches, size_t *dev_bytes)
{
    wavelet_prepare(tab, r);
    const int m = r.shape.n_internal;
    if (m == 0) return;
    wavelet_alloc(st, r);
    std::vector<uint64_t *> ptrs(m);
    for (int v = 0; v < m; ++v) ptrs[v] = reinterpret_cast<uint64_t *>(r.d_sections + r.off_data[v]);
    const size_t scratch = wavelet_fill_bits(st, d_seq, n, r.shape, ptrs, std::vector<uint64_t>(), r.d_ch, launches);
    wavelet_ranks(st, r, launches);
    if (dev_bytes) *dev_bytes = r.section_bytes + m + scratch;
}

// ---- wavelet tree built by several GPUs ---------------------------------------------------------
// GPU r holds slice r of the BWT.  hist_all[r][c] = occurrences of byte c in slice r, so the number of
// members of node v in slice r, and with it the global bit offset of slice r's contribution to node v,
// follow for every (r, v) without looking at any data.  GPU r builds its contributions ("pieces")
// already shifted to their global bit offset modulo 64, so that the assembling GPU only copies words
// (and ORs the shared boundary words).
struct PiecePlan {
    std::vector<uint64_t> count, bit_off, words, word_off; // [world][m]
    std::vector<uint64_t> rank_words, rank_bytes, rank_byte_off; // [world]
    uint64_t total_bytes = 0;
};

PiecePlan plan_pieces(const WtShape &shape, const uint64_t *hist_all, uint32_t world)
{
    const int m = shape.n_internal;
    PiecePlan p;
    p.count.assign((size_t)world * m, 0);
    p.bit_off.assign((size_t)world * m, 0);
    p.words.assign((size_t)world * m, 0);
    p.word_off.assign((size_t)world * m, 0);
    p.rank_words.assign(world, 0);
    p.rank_bytes.assign(world, 0);
    p.rank_byte_off.assign(world, 0);
    for (int v = 0; v < m; ++v) {
        uint64_t run = 0;
        for (uint32_t r = 0; r < world; ++r) {
            uint64_t c = 0;
            for (int s = 0; s < 256; ++s)
                if (shape.info[(size_t)v * 256 + s] & 1u) c += hist_all[(size_t)r * 256 + s];
            p.count[(size_t)r * m + v] = c;
            p.bit_off[(size_t)r * m + v] = run;
            p.words[(size_t)r * m + v] = c ? div_up((run & 63) + c, 64) : 0;
            run += c;
        }
    }
    for (uint32_t r = 0; r < world; ++r) {
        uint64_t w = 0;
        for (int v = 0; v < m; ++v) {
            p.word_off[(size_t)r * m + v] = w;
            w += p.words[(size_t)r * m + v];
        }
        p.rank_words[r] = w;
        p.rank_bytes[r] = w * 8 + align8((size_t)(m ? m : 1)); // words, then the first member symbol of every node
        p.rank_byte_off[r] = p.total_bytes;
        p.total_bytes += p.rank_bytes[r];
    }
    return p;
}

// One bit vector cut into contiguous per-builder ranges: this builder holds bits [o, o + c) of a vector of `nbits`
// bits (a wavelet-tree node, or a section of the .sa file).  On the device its bits start at local bit `base` of an
// array that begins at the superblock holding bit o (word G0 = 4 * (o / 256)), so that local superblocks are global
// superblocks.  `dirs`: a BitRank with Rs / Rb directories; without them (a BlockArray) the words alone.  `last`: no
// later builder has bits of the vector.  The ownership rules are those of the comment above dsmfm_pieces_build.
struct VecPiece {
    uint64_t o = 0, c = 0, nbits = 0;
    bool last = false, dirs = true;
    uint64_t G0 = 0, base = 0, nb = 0, words = 0, nsb = 0, nrb = 0;
    uint64_t off_data = 0, off_rs = 0, off_rb = 0; // offsets of the local arrays in the builder's blob
};

VecPiece vec_layout(uint64_t o, uint64_t c, uint64_t nbits, bool last, bool dirs, size_t &blob)
{
    VecPiece l;
    l.o = o;
    l.c = c;
    l.nbits = nbits;
    l.last = last;
    l.dirs = dirs;
    l.G0 = 4 * (o / 256);
    l.base = o - 64 * l.G0;
    l.nb = l.base + c;
    l.words = l.nb / 64 + 1;
    l.nsb = dirs ? l.nb / 256 + 1 : 0;
    l.nrb = dirs ? l.nb / 64 + 1 : 0;
    l.off_data = blob; blob += l.words * 8;
    l.off_rs = blob;   blob += l.nsb * 8;
    l.off_rb = blob;   blob += align8(l.nrb);
    return l;
}

// `ready`: a page-locked buffer of at least section_bytes acquired ahead of time (or nullptr)
void wavelet_fetch(cudaStream_t st, WaveletResult &r, uint8_t *ready = nullptr)
{
    const int m = r.shape.n_internal;
    if (m > 0) {
        r.h_sections = ready ? ready : static_cast<uint8_t *>(g_pinned.get(r.section_bytes));
        r.h_ch.resize(m);
        DSM_CUDA(cudaMemcpyAsync(r.h_sections, r.d_sections, r.section_bytes, cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaMemcpyAsync(r.h_ch.data(), r.d_ch, (size_t)m, cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaStreamSynchronize(st));
    }
    for (size_t i = 0; i < r.shape.nodes.size(); ++i) {
        const int v = r.shape.internal_of_node[i];
        if (v < 0) continue;
        dsmfm_node &nd = r.shape.nodes[i];
        nd.ch = r.h_ch[v];
        nd.data = reinterpret_cast<const uint64_t *>(r.h_sections + r.off_data[v]);
        nd.Rs = reinterpret_cast<const uint64_t *>(r.h_sections + r.off_rs[v]);
        nd.Rb = r.h_sections + r.off_rb[v];
    }
}

} // namespace

// ---------------------------------------------------------------------------
// the builder handle
// ---------------------------------------------------------------------------
struct dsmfm_builder {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint32_t samplerate = DSMFM_DEFAULT_SAMPLERATE;
    uint32_t flags = 0;
    uint64_t expected = 0;
    uint32_t shard_index = 0, shard_count = 1, shard_span = 1;
    uint64_t shard_rank_begin = 0, shard_m = 0;
    bool assembled = false;
    std::string err;

    // host staging for dsmfm_append (pinned, double buffered)
    static constexpr size_t kStage = 64u << 20;
    uint8_t *stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_free[2] = {nullptr, nullptr};
    int cur = 0;
    size_t cur_used = 0;

    // text in HBM while it streams in
    struct Chunk { uint8_t *d; size_t cap, used; };
    std::vector<Chunk> chunks;
    uint64_t n = 0;

    bool finished = false, built = false, fetched = false;
    bool sealed = false; // dsmfm_block_stats has been taken: no more appends

    // device state of the build
    uint8_t *d_raw = nullptr;
    bool raw_is_chunk = false;
    uint32_t *d_sa = nullptr;      // suffix array of the slice, low position bits (DSMFM_FLAG_KEEP_SA)
    uint8_t *d_sa_hi = nullptr;    // wide builds: position = d_sa_hi << pos_lo_bits | d_sa
    int pos_lo_bits = 32;
    uint32_t *d_doc_end = nullptr; // text position of every document's terminator (DSMFM_FLAG_KEEP_SA, unsharded)
    std::vector<uint8_t> sa_image; // bytes of the .sa file, built on first use
    uint8_t *d_bwt = nullptr;      // lives in the first key buffer of the sort
    WaveletResult wt;
    uint8_t *h_bwt = nullptr;

    uint64_t counts[256];
    dsmfm_index index;
    dsmfm_stats stats;
    size_t dev_now = 0, dev_peak = 0;

    int fail(int code, const char *fmt, ...)
    {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
    int fail_cuda(const CudaError &e)
    {
        return fail(e.code == cudaErrorMemoryAllocation ? DSMFM_ENOMEM : DSMFM_ECUDA, "CUDA error %d (%s) in %s at %s:%d",
                    (int)e.code, cudaGetErrorString(e.code), e.what, e.file, e.line);
    }

    // every device allocation of the builder is tracked so that a failed build leaks nothing
    std::vector<std::pair<void *, size_t>> allocs;
    // DSMFM_GUARD=1 (tests; compute-sanitizer is closed on the pool this was developed on): every device buffer of
    // the builder gets 4 KB of pattern in front and behind, checked when it is released -- a kernel that writes
    // outside its buffer is reported (dsmfm_dbg_guard_violations) instead of silently corrupting a neighbour.
    static constexpr size_t kGuard = 4096;
    static bool guard_on()
    {
        static const bool on = std::getenv("DSMFM_GUARD") != nullptr;
        return on;
    }
    void *dmalloc(size_t bytes)
    {
        const bool g = guard_on();
        uint8_t *raw = static_cast<uint8_t *>(dev_alloc(bytes + (g ? 2 * kGuard : 0), stream));
        if (g) {
            DSM_CUDA(cudaMemsetAsync(raw, 0xA5, kGuard, stream));
            DSM_CUDA(cudaMemsetAsync(raw + kGuard + bytes, 0xA5, kGuard, stream));
        }
        void *p = raw + (g ? kGuard : 0);
        allocs.emplace_back(p, bytes);
        dev_now += bytes;
        dev_peak = std::max(dev_peak, dev_now);
        return p;
    }
    void check_guard(void *p, size_t bytes)
    {
        uint8_t h[2 * kGuard];
        uint8_t *raw = static_cast<uint8_t *>(p) - kGuard;
        if (cudaStreamSynchronize(stream) != cudaSuccess || cudaMemcpy(h, raw, kGuard, cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(h + kGuard, raw + kGuard + bytes, kGuard, cudaMemcpyDeviceToHost) != cudaSuccess)
            return; // (a failed stream: the error is reported where it happened)
        for (size_t i = 0; i < 2 * kGuard; ++i)
            if (h[i] != 0xA5) {
                std::fprintf(stderr, "[dsmfm guard] write outside a %zu-byte device buffer: %s it, offset %zu\n", bytes,
                             i < kGuard ? "in front of" : "behind", i < kGuard ? kGuard - i : i - kGuard);
                ++g_guard_violations;
                break;
            }
    }
    void free_one(void *p, size_t bytes)
    {
        if (guard_on()) {
            check_guard(p, bytes);
            dev_free(static_cast<uint8_t *>(p) - kGuard, stream);
        } else {
            dev_free(p, stream);
        }
    }
    void dfree(void *p)
    {
        if (!p) return;
        for (size_t i = 0; i < allocs.size(); ++i) {
            if (allocs[i].first != p) continue;
            dev_now -= std::min(dev_now, allocs[i].second);
            const size_t bytes = allocs[i].second;
            allocs.erase(allocs.begin() + i);
            free_one(p, bytes);
            return;
        }
    }

    void push_device(const void *src, size_t bytes, cudaMemcpyKind kind)
    {
        pipeline_abandon(); // (text behind a streamed batch: plain statistics at build time)
        const uint8_t *s = static_cast<const uint8_t *>(src);
        while (bytes) {
            if (chunks.empty() || chunks.back().used == chunks.back().cap) {
                size_t cap = chunks.empty() && expected ? (size_t)expected + 64 : (size_t)256 << 20;
                if (cap < bytes && chunks.empty() && !expected) cap = bytes + 64;
                Chunk c{static_cast<uint8_t *>(dmalloc(cap)), cap, 0};
                chunks.push_back(c);
            }
            Chunk &c = chunks.back();
            const size_t take = std::min(bytes, c.cap - c.used);
            DSM_CUDA(cudaMemcpyAsync(c.d + c.used, s, take, kind, stream));
            c.used += take;
            s += take;
            bytes -= take;
            n += take;
        }
    }

    void flush_stage()
    {
        if (!cur_used) return;
        push_device(stage[cur], cur_used, cudaMemcpyHostToDevice);
        DSM_CUDA(cudaEventRecord(stage_free[cur], stream));
        cur ^= 1;
        cur_used = 0;
        DSM_CUDA(cudaEventSynchronize(stage_free[cur])); // the other buffer's copy has drained
    }

    void release_device()
    {
        if (host_prefetch.joinable()) {
            host_prefetch.join();
            g_pinned.put(host_ready);
            host_ready = nullptr;
        }
        for (auto &a : allocs) free_one(a.first, a.second);
        allocs.clear();
        chunks.clear();
        g_pinned.put(ph.h_blob);
        ph.h_blob = nullptr;
        delete ext;
        ext = nullptr;
        for (cudaEvent_t e : pl.ev) cudaEventDestroy(e);
        pl.ev.clear();
        if (pl.copy) cudaStreamDestroy(pl.copy);
        pl = Pipeline();
        d_raw = nullptr;
        d_sa = nullptr;
        d_sa_hi = nullptr;
        d_bwt = nullptr;
        d_doc_end = nullptr;
        sah.d_doc_end = sah.d_sampled = sah.d_ends = nullptr;
        dev_now = 0;
        wt.release(stream);
    }

    // ---- one collection over several builders, packed-text exchange (dsmfm_block_* / dsmfm_build_packed) ----
    // `ext` set: the text to index is a caller-owned row of packed slots (one per block of documents, every
    // builder holds the whole row); this builder's own raw block has been packed into it and released.
    struct PackedText {
        const uint64_t *text = nullptr; // device: world * slot_words (+ 8 zero) words
        SelGeom geom;                   // slot_words, world, symbols per block
        uint64_t n_real = 0;            // symbols of the collection
        uint64_t words = 0;             // world * slot_words
        uint64_t documents = 0, maxlen = 0;
        std::vector<unsigned long long> top; // 4096 bins: top 12 key bits of every suffix of the collection
    };
    PackedText *ext = nullptr;
    bool block_stats_done = false;
    dsmfm_block_info block_info;
    // pieces of the wavelet tree owned by this builder (dsmfm_pieces_build): host copies and their description
    struct PieceHost {
        std::vector<dsmfm_piece> piece;
        std::vector<dsmfm_piece_edge> edge;
        std::vector<VecPiece> vec;                // per internal node
        uint8_t *h_blob = nullptr;                // pinned
        size_t h_bytes = 0;
        uint8_t *d_blob = nullptr;                // device pieces until dsmfm_pieces_fetch
        size_t blob_bytes = 0, ch_off = 0;
        bool built = false;
        std::vector<uint32_t> node_of;
        uint32_t world = 0, rank = 0;
        bool merged = false;
        WtShape shape;
        std::vector<uint64_t> file_off_data, file_off_rs, file_off_rb, file_off_node; // per internal node / per node
        uint64_t file_bytes = 0;
    } ph;
    // .sa samples of a packed-text build with DSMFM_FLAG_KEEP_SA (dsmfm_sa_*): what build() derives from the text and
    // the BWT while both are there, then this builder's share of the five bit vectors of the file
    struct SaHost {
        bool ready = false;              // derived by build()
        uint64_t *d_doc_end = nullptr;   // padded position of every terminator of the collection (u64, document order)
        uint64_t *d_sampled = nullptr;   // the slice's `sampled` bits, laid out as VecPiece of (rank_begin, count)
        uint64_t *d_ends = nullptr;      // bit p: BWT[p] == 0 (end markers of the slice), from bit 0
        uint64_t slot_syms = 0;          // symbols per slot of the packed text
        uint32_t world = 0;
        dsmfm_sa_info info;
        bool built = false, merged = false;
        uint32_t rank = 0;
        uint64_t samples = 0;            // of the whole collection
        unsigned wlen = 0, wdoc = 0;
        VecPiece vec[DSMFM_SA_VECTORS];  // sampled, suffixes, suffixDocId, textLength, Doc
        dsmfm_piece piece[DSMFM_SA_VECTORS];
        dsmfm_piece_edge edge[DSMFM_SA_VECTORS];
        std::vector<uint8_t> h_blob;
    } sah;

    // ---- a text that streams in from host memory (dsmfm_append_batch of a whole collection) ----
    // The copy runs in pieces on a stream of its own; while piece k+1 crosses PCIe the build stream already
    // histograms, scans, packs and keys piece k -- everything of the build that needs no more than the text
    // seen so far.  The alphabet (bits per symbol, code map) is only known at the end, so the pack is SPECULATIVE:
    // it assumes the symbols of the first piece are all there are; build() checks and redoes it otherwise.
    struct Pipeline {
        bool active = false;
        cudaStream_t copy = nullptr;
        std::vector<cudaEvent_t> ev;
        uint64_t *d_counts = nullptr;
        ChunkStat *d_stat = nullptr;
        uint64_t nstat = 0, piece = 0;
        // speculative products
        bool spec = false;
        int bits = 0, first_syms = 0;
        bool carry = false;
        uint8_t code_map[256];
        uint64_t *d_packed = nullptr, *d_keys = nullptr, *d_hist = nullptr;
        uint8_t *d_map = nullptr;
        uint64_t nwords = 0;
    } pl;
    bool append_pipelined(const uint8_t *src, size_t bytes);
    void pipeline_finish_stats(); // waits for the copies, fills block_info
    void pipeline_drop_spec();    // frees the speculative buffers
    void pipeline_abandon();      // more text arrives after all: plain statistics at build time

    uint32_t pre_launches = 0; // kernels launched before build() (the FASTA front end)
    // Page-locking the host buffer of the sections costs ~0.4 s per GB the first time (later builds find it in
    // the pool): a helper thread does it while the GPU sorts, as soon as the histogram fixes the size.
    std::thread host_prefetch;
    uint8_t *host_ready = nullptr;
    size_t host_ready_bytes = 0;
    void append_fasta(const uint8_t *text, size_t m, dsmfm_fasta_info *info);
    void gather_raw();
    void block_stats(uint32_t *L);
    void build();
    void fetch();
    void make_sa_image();
    void sa_derive(int bits, uint32_t *L);
};

// ---------------------------------------------------------------------------
// FASTA front end (fasta.cu): `m` bytes of whole lines -> documents appended to the collection
// ---------------------------------------------------------------------------
void dsmfm_builder::append_fasta(const uint8_t *text, size_t m, dsmfm_fasta_info *info)
{
    cudaStream_t st = stream;
    uint32_t *L = &pre_launches;
    trace("append_fasta: begin");
    pipeline_abandon();
    std::lock_guard<std::mutex> arena_lock(g_fasta_arena.mu);
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    // part 1 (sizes follow the text), part 2 (sizes follow the number of records, known after the first pass)
    const uint64_t ntiles = fasta_tiles(m);
    const size_t o_text = 0, o_last = o_text + up(m + 64), o_entry = o_last + up(ntiles * 8), o_cs = o_entry + up(ntiles * 8),
                 o_ch = o_cs + up(ntiles * 4), o_os = o_ch + up(ntiles * 4), o_oh = o_os + up(ntiles * 8),
                 o_tot = o_oh + up(ntiles * 8), o_cnt = o_tot + 256, part1 = o_cnt + 256;
    uint8_t *base = static_cast<uint8_t *>(g_fasta_arena.reserve(device, std::max(part1, g_fasta_arena.hint[device])));
    uint8_t *d_text = base + o_text;
    long long *d_last = reinterpret_cast<long long *>(base + o_last), *d_entry = reinterpret_cast<long long *>(base + o_entry);
    uint32_t *d_cs = reinterpret_cast<uint32_t *>(base + o_cs), *d_ch = reinterpret_cast<uint32_t *>(base + o_ch);
    uint64_t *d_os = reinterpret_cast<uint64_t *>(base + o_os), *d_oh = reinterpret_cast<uint64_t *>(base + o_oh);
    uint64_t *d_tot = reinterpret_cast<uint64_t *>(base + o_tot);
    unsigned long long *d_cnt = reinterpret_cast<unsigned long long *>(base + o_cnt);
    DSM_CUDA(cudaMemcpyAsync(d_text, text, m, cudaMemcpyHostToDevice, st));
    launch_fasta_scan_lines(st, d_text, m, d_last, d_entry, d_cs, d_ch, d_os, d_oh, d_tot, L);
    uint64_t tot[2] = {0, 0};
    DSM_CUDA(cudaMemcpyAsync(tot, d_tot, sizeof tot, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    const uint64_t nseq = tot[0], nhdr = tot[1], nrec = nhdr + 1;
    trace("append_fasta: text on the device, lines scanned");

    const uint64_t rtiles = fasta_rec_tiles(nrec);
    const size_t bm_bytes = (size_t)div_up(nrec, 32) * 4;
    const size_t o_B = 0, o_O = o_B + up((nrec + 1) * 8), o_rc = o_O + up(nrec * 8), o_ro = o_rc + up(rtiles * 4),
                 o_bm = o_ro + up(rtiles * 8), part2 = o_bm + up(bm_bytes);
    g_fasta_arena.hint[device] = part1 + part2;
    uint8_t *base2 = base + part1;
    void *own2 = nullptr; // the arena was sized for another input: part 2 gets an allocation of its own this time
    if (g_fasta_arena.cap[device] < part1 + part2) base2 = static_cast<uint8_t *>(own2 = dmalloc(part2));
    uint64_t *d_B = reinterpret_cast<uint64_t *>(base2 + o_B), *d_O = reinterpret_cast<uint64_t *>(base2 + o_O);
    uint32_t *d_rc = reinterpret_cast<uint32_t *>(base2 + o_rc);
    uint64_t *d_ro = reinterpret_cast<uint64_t *>(base2 + o_ro);
    uint32_t *d_bm = reinterpret_cast<uint32_t *>(base2 + o_bm);
    const unsigned long long cnt0[4] = {0, 0, ~0ull, 0};
    const uint64_t zero = 0;
    DSM_CUDA(cudaMemcpyAsync(d_cnt, cnt0, sizeof cnt0, cudaMemcpyHostToDevice, st));
    DSM_CUDA(cudaMemcpyAsync(d_B, &zero, 8, cudaMemcpyHostToDevice, st));
    DSM_CUDA(cudaMemcpyAsync(d_B + nrec, &nseq, 8, cudaMemcpyHostToDevice, st));
    launch_fasta_records(st, d_text, m, d_entry, d_os, d_oh, nrec, d_B, d_O, d_rc, d_ro, d_tot, d_cnt, L);
    DSM_CUDA(cudaMemcpyAsync(tot, d_tot, sizeof tot, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    const uint64_t ndocs = tot[0], doc_bytes = 2 * nseq + 2 * ndocs;

    unsigned long long cnt[4] = {0, 0, ~0ull, 0};
    if (doc_bytes) {
        uint8_t *d_out = static_cast<uint8_t *>(dmalloc(doc_bytes + 64));
        DSM_CUDA(cudaMemsetAsync(d_bm, 0, bm_bytes, st));
        launch_fasta_emit(st, d_text, m, d_entry, d_os, d_oh, d_B, d_O, d_out, d_bm, d_cnt, L);
        chunks.push_back(Chunk{d_out, (size_t)doc_bytes + 64, (size_t)doc_bytes});
        n += doc_bytes;
    }
    DSM_CUDA(cudaMemcpyAsync(cnt, d_cnt, sizeof cnt, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st)); // the arena is idle again
    dfree(own2);
    trace("append_fasta: documents written");
    info->records = nhdr;
    info->documents = ndocs;
    info->bases = nseq;
    info->doc_bytes = doc_bytes;
    info->bad_headers = cnt[0];
    info->invalid_records = cnt[1];
    info->first_invalid_offset = cnt[2];
}

// ---------------------------------------------------------------------------
// host text streaming in: copy pieces on one stream, work on them on the other
// ---------------------------------------------------------------------------
namespace {
constexpr uint64_t kLongKeyAbove = 3500000000ull; // indexed symbols above which the first key is 18 symbols (build())
// Dense codes (0 = terminator, 1..sigma in byte order) of the bytes that occur; returns the bits per symbol.
int alphabet_of(const uint64_t counts[256], uint8_t code_map[256], uint32_t *sigma_out)
{
    std::memset(code_map, 0, 256);
    uint32_t sigma = 0;
    for (int c = 1; c < 256; ++c)
        if (counts[c]) code_map[c] = (uint8_t)++sigma;
    if (sigma_out) *sigma_out = sigma;
    return sigma <= 7 ? 3 : (sigma <= 15 ? 4 : 8);
}

// Symbols of the first key (sorted by the initial radix sort): `first_key_bits` when > 0, else the default of
// build() -- 48 bits, 54 / 56 above kLongKeyAbove indexed symbols, DSMFM_FIRST_KEY_BITS overriding both.
// Widths outside [8, SPW * bits] mean the whole word.
int first_key_syms(int bits, uint64_t n_idx, int first_key_bits)
{
    const int spw = 64 / bits;
    if (first_key_bits <= 0) {
        uint64_t long_key_above = kLongKeyAbove;
        if (const char *e = std::getenv("DSMFM_LONG_KEY_ABOVE")) long_key_above = std::strtoull(e, nullptr, 10);
        first_key_bits = 48;
        if (n_idx > long_key_above) first_key_bits = bits == 3 ? 54 : (bits == 4 ? 56 : 48);
        if (const char *e = std::getenv("DSMFM_FIRST_KEY_BITS")) first_key_bits = std::atoi(e);
    }
    if (first_key_bits < 8 || first_key_bits > spw * bits) first_key_bits = spw * bits;
    return std::max(1, first_key_bits / bits);
}

// first key of an unsharded build: symbols sorted, and whether the BWT symbol rides above them
void first_key_shape(int bits, uint64_t n_idx, int first_key_bits, int *first_syms, bool *carry)
{
    *first_syms = first_key_syms(bits, n_idx, first_key_bits);
    *carry = *first_syms * bits + bits <= 64;
}

// One word range of a text that is packed and keyed piece by piece: packs words [w0, w0 + wn) from `raw`, the
// text from symbol w0 * SPW on (`len` symbols of it; the last range also writes the zero words behind the text),
// then keys every word whose successor is packed by now.  Returns the words keyed so far.
uint64_t pack_and_key_range(cudaStream_t st, int bits, const uint8_t *raw, uint64_t len, const uint8_t *d_map,
                            uint64_t *d_packed, uint64_t w0, uint64_t wn, bool last, uint64_t n, uint64_t *d_keys,
                            int first_syms, bool carry, uint64_t *d_hist, uint64_t keyed_to, uint32_t *L)
{
    launch_pack(st, bits, raw, len, d_map, d_packed + w0, wn, L);
    const uint64_t upto = last ? div_up(n, 64 / bits) : w0 + wn - 1;
    if (upto > keyed_to) {
        launch_make_keys_hist(st, bits, d_packed, n, d_keys, first_syms, carry, d_hist, L, keyed_to, upto);
        keyed_to = upto;
    }
    return keyed_to;
}
} // namespace

bool dsmfm_builder::append_pipelined(const uint8_t *src, size_t bytes)
{
    // pieces of 63 MiB: a multiple of 21, 16 and 8 symbols (whole packed words for 3-, 4- and 8-bit symbols), of the
    // 16-byte vectors the kernels load and of the 16 KiB chunks of the document statistics
    constexpr uint64_t kPiece = 21ull * 3145728ull;
    static_assert(kPiece % 16 == 0 && kPiece % kStatChunk == 0, "piece alignment");
    static const bool off = std::getenv("DSMFM_NO_PIPELINE") != nullptr;
    if (off || n != 0 || !chunks.empty() || cur_used != 0 || shard_count > 1 || (flags & DSMFM_FLAG_KEEP_SA) ||
        bytes < 3 * kPiece || bytes >= (1ull << 32) - 4096)
        return false;
    cudaStream_t st = stream;
    uint32_t *L = &pre_launches;
    uint8_t *d = static_cast<uint8_t *>(dmalloc(bytes + 64));
    chunks.push_back(Chunk{d, bytes + 64, bytes});
    n = bytes;
    if (!pl.copy) DSM_CUDA(cudaStreamCreateWithFlags(&pl.copy, cudaStreamNonBlocking));
    pl.piece = kPiece;
    const uint64_t npiece = div_up(bytes, kPiece);
    pl.ev.resize(npiece);
    for (auto &e : pl.ev) DSM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    // whatever is queued on the build stream (nothing, normally) precedes the copies
    cudaEvent_t start;
    DSM_CUDA(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    DSM_CUDA(cudaEventRecord(start, st));
    DSM_CUDA(cudaStreamWaitEvent(pl.copy, start, 0));
    cudaEventDestroy(start);
    for (uint64_t k = 0; k < npiece; ++k) {
        const uint64_t o = k * kPiece, len = std::min<uint64_t>(kPiece, bytes - o);
        DSM_CUDA(cudaMemcpyAsync(d + o, src + o, len, cudaMemcpyHostToDevice, pl.copy));
        DSM_CUDA(cudaEventRecord(pl.ev[k], pl.copy));
    }
    pl.nstat = div_up(bytes, kStatChunk);
    pl.d_counts = static_cast<uint64_t *>(dmalloc(256 * 8));
    pl.d_stat = static_cast<ChunkStat *>(dmalloc(pl.nstat * sizeof(ChunkStat)));
    DSM_CUDA(cudaMemsetAsync(pl.d_counts, 0, 256 * 8, st));
    auto stats_of = [&](uint64_t k) {
        const uint64_t o = k * kPiece, len = std::min<uint64_t>(kPiece, bytes - o);
        DSM_CUDA(cudaStreamWaitEvent(st, pl.ev[k], 0));
        launch_byte_hist(st, d + o, len, pl.d_counts, L);
        launch_doc_stats(st, d + o, len, pl.d_stat + o / kStatChunk, L); // (positions relative to the piece)
    };
    pl.active = true;
    // the alphabet of the first piece: the guess for the whole text
    stats_of(0);
    uint64_t first_counts[256];
    DSM_CUDA(cudaMemcpyAsync(first_counts, pl.d_counts, sizeof first_counts, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    uint32_t sigma = 0;
    pl.bits = alphabet_of(first_counts, pl.code_map, &sigma);
    first_key_shape(pl.bits, bytes, 0, &pl.first_syms, &pl.carry);
    const int spw = 64 / pl.bits;
    pl.spec = sigma > 0 && (pl.first_syms * pl.bits + 7) / 8 <= kMaxPasses;
    uint64_t text_words = div_up(bytes, (uint64_t)spw);
    if (pl.spec) {
        pl.nwords = text_words + 8;
        pl.d_map = static_cast<uint8_t *>(dmalloc(256));
        pl.d_packed = static_cast<uint64_t *>(dmalloc(pl.nwords * 8));
        pl.d_keys = static_cast<uint64_t *>(dmalloc(bytes * 8));
        pl.d_hist = static_cast<uint64_t *>(dmalloc(sizeof(uint64_t) * kMaxPasses * kRadix));
        DSM_CUDA(cudaMemcpyAsync(pl.d_map, pl.code_map, 256, cudaMemcpyHostToDevice, st));
        DSM_CUDA(cudaMemsetAsync(pl.d_hist, 0, sizeof(uint64_t) * kMaxPasses * kRadix, st));
    }
    uint64_t keyed_to = 0; // words whose keys are built
    for (uint64_t k = 0; k < npiece; ++k) {
        if (k) stats_of(k);
        if (!pl.spec) continue;
        const uint64_t o = k * kPiece, len = std::min<uint64_t>(kPiece, bytes - o);
        const bool last = k + 1 == npiece;
        const uint64_t w0 = o / spw, wn = last ? pl.nwords - w0 : len / spw;
        keyed_to = pack_and_key_range(st, pl.bits, d + o, len, pl.d_map, pl.d_packed, w0, wn, last, bytes, pl.d_keys,
                                      pl.first_syms, pl.carry, pl.d_hist, keyed_to, L);
    }
    return true;
}

void dsmfm_builder::pipeline_finish_stats()
{
    cudaStream_t st = stream;
    std::memset(&block_info, 0, sizeof block_info);
    block_info.bytes = n;
    std::vector<ChunkStat> hstat(pl.nstat);
    DSM_CUDA(cudaMemcpyAsync(block_info.counts, pl.d_counts, 256 * 8, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(hstat.data(), pl.d_stat, pl.nstat * sizeof(ChunkStat), cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st)); // every piece has arrived and has been looked at
    dfree(pl.d_counts);
    dfree(pl.d_stat);
    pl.d_counts = nullptr;
    pl.d_stat = nullptr;
    uint64_t maxgap = 0, mingap = ~0ull;
    int64_t prev = -1, lastz = -1;
    const uint64_t per_piece = pl.piece / kStatChunk;
    for (uint64_t i = 0; i < pl.nstat; ++i) {
        const ChunkStat &c = hstat[i];
        if (c.last < 0) continue;
        const int64_t base = (int64_t)((i / per_piece) * pl.piece); // the kernel saw the piece, not the text
        const uint64_t g = (uint64_t)(c.first + base - prev);
        maxgap = std::max(maxgap, g);
        mingap = std::min(mingap, g);
        maxgap = std::max(maxgap, c.maxgap);
        mingap = std::min(mingap, c.mingap);
        prev = c.last + base;
        lastz = c.last + base;
    }
    pl.active = false;
    block_stats_done = true;
    if (lastz != (int64_t)n - 1)
        throw CudaError{cudaErrorInvalidValue, "text does not end with a document terminator", __FILE__, __LINE__};
    block_info.documents = block_info.counts[0];
    block_info.max_text_length = maxgap;
    block_info.empty_document = mingap == 1 ? 1u : 0u;
}

void dsmfm_builder::pipeline_drop_spec()
{
    if (pl.d_packed) dfree(pl.d_packed);
    if (pl.d_keys) dfree(pl.d_keys);
    if (pl.d_hist) dfree(pl.d_hist);
    if (pl.d_map) dfree(pl.d_map);
    pl.d_packed = pl.d_keys = pl.d_hist = nullptr;
    pl.d_map = nullptr;
    pl.spec = false;
}

void dsmfm_builder::pipeline_abandon()
{
    if (!pl.active) return;
    DSM_CUDA(cudaStreamSynchronize(pl.copy));
    DSM_CUDA(cudaStreamSynchronize(stream));
    pipeline_drop_spec();
    dfree(pl.d_counts);
    dfree(pl.d_stat);
    pl.d_counts = nullptr;
    pl.d_stat = nullptr;
    pl.active = false;
}

// ---------------------------------------------------------------------------
// the raw text in one piece; its statistics
// ---------------------------------------------------------------------------
void dsmfm_builder::gather_raw()
{
    if (d_raw) return;
    cudaStream_t st = stream;
    if (chunks.size() == 1) {
        d_raw = chunks[0].d;
        raw_is_chunk = true;
        return;
    }
    d_raw = static_cast<uint8_t *>(dmalloc(n + 64));
    raw_is_chunk = false;
    size_t o = 0;
    for (auto &c : chunks) {
        DSM_CUDA(cudaMemcpyAsync(d_raw + o, c.d, c.used, cudaMemcpyDeviceToDevice, st));
        o += c.used;
    }
    DSM_CUDA(cudaStreamSynchronize(st));
    for (auto &c : chunks) dfree(c.d);
    chunks.clear();
}

// 256-bin histogram (= the BWT's counts: C[] and the Huffman weights), number of documents, longest document
// incl. its terminator (TextCollectionBuilder.cpp:73-81), empty-document detection.  Synchronises the stream.
void dsmfm_builder::block_stats(uint32_t *L)
{
    cudaStream_t st = stream;
    std::memset(&block_info, 0, sizeof block_info);
    block_info.bytes = n;
    block_stats_done = true;
    if (n == 0) return;
    uint64_t *d_counts = static_cast<uint64_t *>(dmalloc(256 * 8));
    const uint64_t nstat = div_up(n, kStatChunk);
    ChunkStat *d_stat = static_cast<ChunkStat *>(dmalloc(nstat * sizeof(ChunkStat)));
    DSM_CUDA(cudaMemsetAsync(d_counts, 0, 256 * 8, st));
    launch_byte_hist(st, d_raw, n, d_counts, L);
    launch_doc_stats(st, d_raw, n, d_stat, L);
    std::vector<ChunkStat> hstat(nstat);
    DSM_CUDA(cudaMemcpyAsync(block_info.counts, d_counts, 256 * 8, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(hstat.data(), d_stat, nstat * sizeof(ChunkStat), cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    dfree(d_counts);
    dfree(d_stat);

    uint64_t maxgap = 0, mingap = ~0ull;
    int64_t prev = -1, lastz = -1;
    for (const ChunkStat &c : hstat) {
        if (c.last < 0) continue;
        const uint64_t g = (uint64_t)(c.first - prev);
        maxgap = std::max(maxgap, g);
        mingap = std::min(mingap, g);
        maxgap = std::max(maxgap, c.maxgap);
        mingap = std::min(mingap, c.mingap);
        prev = c.last;
        lastz = c.last;
    }
    if (lastz != (int64_t)n - 1)
        throw CudaError{cudaErrorInvalidValue, "text does not end with a document terminator", __FILE__, __LINE__};
    block_info.documents = block_info.counts[0];
    block_info.max_text_length = maxgap;
    block_info.empty_document = mingap == 1 ? 1u : 0u;
}

// ---------------------------------------------------------------------------
// the device build
// ---------------------------------------------------------------------------
void dsmfm_builder::build()
{
    cudaStream_t st = stream;
    uint32_t *L = &stats.kernel_launches;
    std::memset(&stats, 0, sizeof stats);
    cudaEvent_t ev[8];
    for (auto &e : ev) DSM_CUDA(cudaEventCreate(&e));
    cudaEvent_t ev_pass0, ev_pass1;
    DSM_CUDA(cudaEventCreate(&ev_pass0));
    DSM_CUDA(cudaEventCreate(&ev_pass1));

    trace("build: begin");
    const bool packed_in = ext != nullptr;
    bool empty_collection = false;
    uint64_t maxgap = 0;
    if (!packed_in) {
        flush_stage();
        if (n == 0) { // TextCollectionBuilder.cpp:111-119: one empty text
            const uint8_t z = 0;
            push_device(&z, 1, cudaMemcpyHostToDevice);
            DSM_CUDA(cudaStreamSynchronize(st));
            empty_collection = true;
        }
    }

    // Random 16-byte gathers from the packed text dominate the refinement's DRAM traffic; with the default
    // 64-byte L2 fetch granularity every miss drags in a second, unused sector.  The limit is a property of the
    // device context, so it is set ONCE per device by the first build of the process (not per build, and not
    // restored: toggling it around every build would change device-global state under other streams' feet).
    // DSMFM_L2_FETCH=0 leaves the limit alone, any other value overrides the 32 bytes.
    {
        static DeviceOnce gran_once;
        gran_once.run([] {
            size_t want_gran = 32;
            if (const char *e = std::getenv("DSMFM_L2_FETCH")) want_gran = (size_t)std::atoi(e);
            if (want_gran) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, want_gran);
        });
    }

    DSM_CUDA(cudaEventRecord(ev[0], st));
    if (!packed_in) {
        // ---- contiguous text, histogram, document statistics ----------------------------------
        if (pl.active) pipeline_finish_stats(); // a streamed batch: its pieces were looked at as they arrived
        gather_raw();
        if (!block_stats_done) block_stats(L);
        std::memcpy(counts, block_info.counts, sizeof counts);
        maxgap = block_info.max_text_length;
        if (block_info.empty_document && !empty_collection)
            throw CudaError{cudaErrorInvalidValue, "EMPTY", __FILE__, __LINE__};
    } else {
        maxgap = ext->maxlen;
    }
    const uint64_t n_idx = packed_in ? ext->n_real : n;                                // symbols of the index

    uint8_t code_map[256];
    uint32_t sigma = 0;
    const int bits = alphabet_of(counts, code_map, &sigma);
    const int spw = 64 / bits;
    // positions are positions in the text as it lies in HBM: the packed slots with their padding when the text
    // came in packed (one slot per block), the plain text otherwise
    const uint64_t n_text = packed_in ? ext->words * (uint64_t)spw : n;
    // The initial radix sort orders suffixes by their first `first_syms` symbols only (48 key bits = 6
    // LSD passes instead of 8); the refinement rounds extend from there.  For DNA reads 16 symbols
    // already separate everything that is not a genuine repeat, so the two saved passes cost almost
    // no extra refinement work.  That stops being true when the collection is large: with L distinct loci the
    // chance that a 16-mer also occurs at an unrelated locus is about L / 4^16, and unrelated loci in one tie
    // group carry different BWT symbols, so the group has to be refined (8 GPUs x 1 Gbp: 3.2 G loci, 75 %;
    // the refinement took 75 ms per GPU instead of 24).  Collections beyond 3.5 G symbols therefore sort 18
    // symbols (54 bits, a seventh pass of 6 bits): 16x fewer chance matches for about 13 ms of sorting.  (The
    // threshold sits between the 1 Gbp sample -- 2.02 G symbols, where the seventh pass costs what it saves -- and two
    // of them, 4.04 G, where the refinement takes 36 ms with 16 symbols.)
    // DSMFM_FIRST_KEY_BITS overrides (any multiple of bits/symbol); DSMFM_LONG_KEY_ABOVE moves the threshold (tests).
    int first_syms = first_key_syms(bits, n_idx, 0);
    // Text positions: the u32 value of the sort holds the low `lo_bits` bits (32; fewer only in tests, which
    // thereby exercise the wide path on small inputs), anything above rides in the key's spare top bits.
    // A packed-text build always takes the key-range path (its padding positions must not be sorted).
    const bool sharded = shard_count > 1 || packed_in;
    int lo_bits = 32;
    if (const char *e = std::getenv("DSMFM_POS_LO_BITS")) lo_bits = std::min(32, std::max(4, std::atoi(e)));
    if (!sharded) lo_bits = 32;
    int hi_bits = 0;
    while (lo_bits + hi_bits < 64 && ((n_text - 1) >> (lo_bits + hi_bits))) ++hi_bits;
    const bool wide = hi_bits > 0;
    if (wide && !sharded)
        throw CudaError{cudaErrorInvalidValue, "more than 2^32 symbols in one unsharded build (set shard_count / shard_span)", __FILE__, __LINE__};
    if (hi_bits > 8)
        throw CudaError{cudaErrorInvalidValue, "more than 2^32 * 256 symbols", __FILE__, __LINE__};
    // sharded builds always carry the BWT symbol (and the high position bits) above the sorted key bits
    if (sharded)
        while (first_syms > 1 && first_syms * bits + bits + hi_bits > 64) --first_syms;
    const bool carry_bwt = first_syms * bits + bits + hi_bits <= 64;
    if (sharded && !carry_bwt)
        throw CudaError{cudaErrorInvalidValue, "no room in the key for the carried fields", __FILE__, __LINE__};
    uint8_t inv_map[256];
    std::memset(inv_map, 0, sizeof inv_map);
    for (int c = 1; c < 256; ++c)
        if (code_map[c]) inv_map[code_map[c]] = (uint8_t)c;
    // a streamed batch was packed and keyed with the alphabet of its first piece: keep that work if the guess held
    bool spec_ok = pl.spec && !sharded && !packed_in && pl.bits == bits && pl.first_syms == first_syms &&
                   pl.carry == carry_bwt && std::memcmp(pl.code_map, code_map, sizeof code_map) == 0;
    if (pl.spec && !spec_ok) pipeline_drop_spec();
    stats.streamed = spec_ok ? 1u : 0u;

    if (!sharded && !host_prefetch.joinable()) {
        dsmfm_code tab[256];
        WaveletResult probe;
        if (build_codetable(counts, tab) <= 32) {
            wavelet_prepare(tab, probe);
            if (probe.shape.n_internal > 0) {
                const size_t want = probe.section_bytes;
                const int dev = device;
                host_ready_bytes = want;
                host_prefetch = std::thread([this, want, dev] {
                    cudaSetDevice(dev);
                    try {
                        host_ready = static_cast<uint8_t *>(g_pinned.get(want));
                    } catch (...) {
                        host_ready = nullptr;
                        host_ready_bytes = 0;
                    }
                });
            }
        }
    }
    index.n = n_idx;
    index.samplerate = samplerate;
    index.number_of_texts = (uint32_t)counts[0];
    index.max_text_length = maxgap;
    stats.n = n_idx;
    stats.bases = n_idx - counts[0];
    stats.bits_per_symbol = bits;
    stats.sigma = sigma;

    // ---- pack -----------------------------------------------------------------------
    // zero words behind the text: refinement rows read up to 5 words ahead
    const uint64_t nwords = packed_in ? ext->words + 8 : div_up(n, spw) + 8;
    uint8_t *d_map = static_cast<uint8_t *>(dmalloc(256));
    uint8_t *d_inv = static_cast<uint8_t *>(dmalloc(256));
    DSM_CUDA(cudaMemcpyAsync(d_inv, inv_map, 256, cudaMemcpyHostToDevice, st));
    DSM_CUDA(cudaMemcpyAsync(d_map, code_map, 256, cudaMemcpyHostToDevice, st));
    uint64_t *d_packed = nullptr;
    if (packed_in) {
        d_packed = const_cast<uint64_t *>(ext->text);
    } else if (spec_ok) {
        d_packed = pl.d_packed; // packed piece by piece while the text streamed in (same words, same zero tail)
        pl.d_packed = nullptr;
        dfree(d_raw);
        chunks.clear();
        d_raw = nullptr;
    } else {
        d_packed = static_cast<uint64_t *>(dmalloc(nwords * 8));
        launch_pack(st, bits, d_raw, n, d_map, d_packed, nwords, L);
        if ((flags & DSMFM_FLAG_KEEP_SA) && shard_count <= 1) { // the .sa writer needs the document boundaries
            d_doc_end = static_cast<uint32_t *>(dmalloc((size_t)counts[0] * 4 + 16));
            uint64_t *d_tile = static_cast<uint64_t *>(dmalloc(term_tiles(n) * 8));
            launch_term_positions(st, d_raw, n, d_tile, d_doc_end, L);
            dfree(d_tile);
        }
        // the raw text is not looked at again: everything downstream reads the packed text (3/8 of its size)
        dfree(d_raw);
        chunks.clear();
        d_raw = nullptr;
    }
    DSM_CUDA(cudaEventRecord(ev[1], st));
    trace("build: statistics done, pack launched");

    // ---- which suffixes this builder sorts ------------------------------------------------
    // Unsharded: all n, in one go.  Sharded: the collection is cut into `shard_count` key ranges of
    // about equal population (from a 4096-bin histogram of the top key bits, which every builder
    // computes identically from the replicated text, so no communication is needed to agree on them);
    // this builder sorts ranges [shard_index, shard_index + shard_span) one after the other, which
    // yields one contiguous slice of the global suffix order and bounds the sort buffers by the
    // largest single range.
    struct Range { uint64_t key_lo, key_hi, count, rank_begin; };
    std::vector<Range> ranges;
    const int key_bits = first_syms * bits; // sorted bits of the first key
    const int hi_shift = wide ? key_bits + bits : 0;
    const int top_bits = key_bits < 12 ? key_bits : 12; // key ranges are cut at multiples of 2^(key_bits - top_bits)
    if (!sharded) {
        ranges.push_back(Range{0, 0, n, 0});
    } else {
        const int nbins = 1 << top_bits;
        std::vector<unsigned long long> top(4096, 0ull);
        if (packed_in) {
            // every builder counted the suffixes of its own block while packing it; the sum came in with the text
            if (top_bits != 12)
                throw CudaError{cudaErrorInvalidValue, "packed-text builds need a first key of >= 12 bits", __FILE__, __LINE__};
            top = ext->top;
        } else {
            unsigned long long *d_top = static_cast<unsigned long long *>(dmalloc(4096 * 8));
            DSM_CUDA(cudaMemsetAsync(d_top, 0, 4096 * 8, st));
            launch_key_top_hist(st, bits, d_packed, n, first_syms, top_bits, d_top, L);
            DSM_CUDA(cudaMemcpyAsync(top.data(), d_top, 4096 * 8, cudaMemcpyDeviceToHost, st));
            DSM_CUDA(cudaStreamSynchronize(st));
            dfree(d_top);
        }
        // range s takes the bins whose running count first reaches s*n/G ... (s+1)*n/G
        std::vector<int> cut(shard_count + 1, nbins);
        cut[0] = 0;
        uint64_t run = 0;
        uint32_t next = 1;
        for (int bin = 0; bin < nbins && next < shard_count; ++bin) {
            run += top[bin];
            while (next < shard_count &&
                   run >= (n_idx / shard_count) * next + (n_idx % shard_count) * next / shard_count) {
                cut[next++] = bin + 1;
            }
        }
        std::vector<uint64_t> before(nbins + 1, 0);
        for (int bin = 0; bin < nbins; ++bin) before[bin + 1] = before[bin] + top[bin];
        for (uint32_t v = shard_index; v < shard_index + shard_span; ++v) {
            const int b_lo = cut[v], b_hi = cut[v + 1];
            Range r;
            r.rank_begin = before[b_lo];
            r.count = before[b_hi] - before[b_lo];
            r.key_lo = (uint64_t)b_lo << (key_bits - top_bits);
            r.key_hi = b_hi >= nbins ? (1ull << key_bits) : ((uint64_t)b_hi << (key_bits - top_bits));
            if (v == shard_index) shard_rank_begin = r.rank_begin;
            if (r.count) ranges.push_back(r);
        }
    }
    uint64_t m_total = 0, m_max = 1;
    for (const Range &r : ranges) {
        m_total += r.count;
        m_max = std::max(m_max, r.count);
    }
    shard_m = m_total;
    if (m_max >= (1ull << 32) - kRefCap - 64)
        throw CudaError{cudaErrorInvalidValue,
                        "more than 2^32 suffixes in one sort range (use more shards: shard_count / shard_span)", __FILE__, __LINE__};

    // ---- buffers of one range (sized for the largest) -------------------------------------
    uint64_t *d_keys_a = spec_ok ? pl.d_keys : static_cast<uint64_t *>(dmalloc(m_max * 8));
    if (spec_ok) pl.d_keys = nullptr;
    uint64_t *d_keys_b = static_cast<uint64_t *>(dmalloc(m_max * 8));
    uint32_t *d_vals_a = static_cast<uint32_t *>(dmalloc(m_max * 4 + 16));
    uint32_t *d_vals_b = static_cast<uint32_t *>(dmalloc(m_max * 4 + 16));
    trace("build: sort buffers allocated");
    RadixWorkspace ws; // buffers owned by the builder's allocation list
    ws.status_tiles = div_up(m_max < kSweepPortion ? m_max : kSweepPortion, kSweepTile);
    ws.hist = static_cast<uint64_t *>(dmalloc(sizeof(uint64_t) * kMaxPasses * kRadix));
    ws.carry = static_cast<uint64_t *>(dmalloc(sizeof(uint64_t) * 2 * kRadix));
    ws.status = static_cast<uint32_t *>(dmalloc(sizeof(uint32_t) * ws.status_tiles * kRadix));
    ws.counter = static_cast<uint32_t *>(dmalloc(sizeof(uint32_t)));
    SelGeom sel_geom;
    std::memset(&sel_geom, 0, sizeof sel_geom);
    if (packed_in) {
        sel_geom = ext->geom;
    } else {
        sel_geom.slot_words = nwords - 8;
        sel_geom.world = 1;
        sel_geom.bytes[0] = n;
    }
    uint32_t *d_sel_lut = sharded ? static_cast<uint32_t *>(dmalloc(sizeof(uint32_t) * kSelLutWords)) : nullptr;
    const int full_key_bits = spw * bits; // sorted bits of a refinement key (large-group path)
    const uint64_t hwords = head_words_for(m_max);
    uint32_t *d_head[2];
    d_head[0] = static_cast<uint32_t *>(dmalloc(hwords * 4));
    d_head[1] = static_cast<uint32_t *>(dmalloc(hwords * 4));
    uint32_t *d_diff = static_cast<uint32_t *>(dmalloc(hwords * 4)); // see launch_heads
    // [0,64): suffixes left in groups of >= 2; [64,128): keys the refinement gathered from the text
    unsigned long long *d_remaining = static_cast<unsigned long long *>(dmalloc(128 * 8));
    const uint32_t big_cap = (uint32_t)(m_max / kRefGroupMaxWarps + 2);
    uint32_t *d_big_heads = static_cast<uint32_t *>(dmalloc((size_t)big_cap * 4));
    uint32_t *d_big_len = static_cast<uint32_t *>(dmalloc((size_t)big_cap * 4));
    uint32_t *d_big_count = static_cast<uint32_t *>(dmalloc(4));
    const uint32_t nwin_max = (uint32_t)div_up(m_max, kRefWindow);
    uint32_t *d_win_flag = static_cast<uint32_t *>(dmalloc((size_t)nwin_max * 4));
    uint32_t *d_win_list[2];
    d_win_list[0] = static_cast<uint32_t *>(dmalloc((size_t)nwin_max * 4));
    d_win_list[1] = static_cast<uint32_t *>(dmalloc((size_t)nwin_max * 4));
    uint32_t *d_win_count = static_cast<uint32_t *>(dmalloc(4));
    // results of the whole slice: the BWT (its own buffer: the key buffers are still needed by the
    // large-group path), optionally the suffix array
    d_bwt = static_cast<uint8_t *>(dmalloc(m_total + 64));
    const bool keep_sa = (flags & DSMFM_FLAG_KEEP_SA) != 0;
    uint32_t *d_sa_all = nullptr;
    uint8_t *d_hi_buf = nullptr; // wide: high parts of the positions (whole slice if kept, else one range)
    if (sharded && keep_sa) d_sa_all = static_cast<uint32_t *>(dmalloc(m_total * 4 + 16));
    if (wide) d_hi_buf = static_cast<uint8_t *>(dmalloc((keep_sa ? m_total : m_max) + 16));

    // multi-step: one launch resolves every group that fits a CTA (DSMFM_REFINE_SINGLE_STEP=1 keeps
    // the one-depth-per-launch schedule, used by the tests to exercise the worklist path)
    bool multi_step = true;
    if (const char *e = std::getenv("DSMFM_REFINE_SINGLE_STEP")) multi_step = std::atoi(e) == 0;
    // The index needs the BWT, not the suffix array: tie groups whose members share one BWT symbol stay unsorted
    // unless the suffix array itself is wanted (DSMFM_FLAG_KEEP_SA; DSMFM_REFINE_FULL_ORDER=1 forces it).
    bool full_order = keep_sa;
    if (const char *e = std::getenv("DSMFM_REFINE_FULL_ORDER")) full_order = full_order || std::atoi(e) != 0;
    int key_words = 1; // symbols compared per step = key_words * SPW (DSMFM_REFINE_KEY_WORDS=2: 128-bit keys)
    if (const char *e = std::getenv("DSMFM_REFINE_KEY_WORDS")) key_words = std::atoi(e) == 2 ? 2 : 1;

    cudaEvent_t evr[3];
    for (auto &e : evr) DSM_CUDA(cudaEventCreate(&e));
    float ms_sort = 0.f, ms_refine = 0.f, ms_passes = 0.f;
    uint64_t pass_launch_bytes = 0;
    uint32_t pass_launches = 0, rounds_max = 0;
    uint32_t *d_last_sorted_vals = nullptr, *d_last_other_vals = nullptr;

    uint64_t off = 0; // slot of the range's first suffix inside this builder's slice
    for (const Range &rg : ranges) {
        const uint64_t m = rg.count;
        uint8_t *bwt_out = d_bwt + off;
        uint8_t *hi_out = wide ? d_hi_buf + (keep_sa ? off : 0) : nullptr;
        DSM_CUDA(cudaEventRecord(evr[0], st));

        // ---- initial sort by the first `first_syms` symbols -------------------------------
        // When the key leaves room, the symbol before each suffix rides above the sorted bits and the
        // BWT falls out of the sort; otherwise it is gathered from the text at the end.
        bool hist_ready = false;
        if (!sharded) {
            // keys and their digit histogram in one pass over the packed text
            if (spec_ok) { // keys and digit counts were made as the pieces arrived
                DSM_CUDA(cudaMemcpyAsync(ws.hist, pl.d_hist, sizeof(uint64_t) * kMaxPasses * kRadix, cudaMemcpyDeviceToDevice, st));
            } else {
                DSM_CUDA(cudaMemsetAsync(ws.hist, 0, sizeof(uint64_t) * kMaxPasses * kRadix, st));
                launch_make_keys_hist(st, bits, d_packed, n, d_keys_a, first_syms, carry_bwt, ws.hist, L);
            }
            hist_ready = true;
        } else {
            const uint64_t twords = nwords - 8; // words that hold text
            const uint64_t ntile = select_tiles(twords, bits, first_syms, top_bits);
            uint64_t *d_tile = static_cast<uint64_t *>(dmalloc(ntile * 8));
            launch_select(st, bits, d_packed, twords, first_syms, top_bits, carry_bwt, rg.key_lo, rg.key_hi, d_tile,
                          ws.counter, d_keys_a, d_vals_a, lo_bits, hi_shift, sel_geom, d_sel_lut, L);
            dfree(d_tile);
        }
        const int passes = radix_sort_pairs(st, ws, d_keys_a, d_vals_a, d_keys_b, d_vals_b, m, 0, key_bits, !sharded, L,
                                            ev_pass0, ev_pass1, hist_ready);
        uint64_t *d_sorted_keys = (passes & 1) ? d_keys_b : d_keys_a;
        uint32_t *d_sorted_vals = (passes & 1) ? d_vals_b : d_vals_a;
        uint32_t *d_other_vals = (passes & 1) ? d_vals_a : d_vals_b;
        d_last_sorted_vals = d_sorted_vals;
        d_last_other_vals = d_other_vals;
        stats.sort_passes = passes;
        pass_launches += (uint32_t)passes * (uint32_t)div_up(m, kSweepPortion); // a pass is one launch per portion
        pass_launch_bytes += (uint64_t)passes * m * 24ull;

        DSM_CUDA(cudaMemsetAsync(d_remaining, 0, 128 * 8, st));
        const uint64_t hw = head_words_for(m);
        const bool use_diff = carry_bwt && !full_order;
        launch_heads(st, bits, d_sorted_keys, m, d_head[0], hw, d_remaining, key_bits, d_inv,
                     carry_bwt ? bwt_out : nullptr, hi_out, hi_shift, use_diff ? d_diff : nullptr, L);
        DSM_CUDA(cudaEventRecord(evr[1], st));

        auto read_remaining = [&]() -> uint64_t {
            unsigned long long h[128];
            DSM_CUDA(cudaMemcpyAsync(h, d_remaining, sizeof h, cudaMemcpyDeviceToHost, st));
            DSM_CUDA(cudaStreamSynchronize(st));
            uint64_t t = 0;
            for (int i = 0; i < 64; ++i) t += h[i];
            for (int i = 64; i < 128; ++i) stats.refine_key_fetches += h[i];
            return t;
        };
        uint64_t remaining = read_remaining();
        trace("build: initial sort done");

        // What the refinement works on: the suffix array itself or, in BWT-only builds, dense copies of the groups
        // whose members carry different BWT symbols (kernels.cu, "compaction of the groups that have to be sorted").
        uint32_t *r_sa = d_sorted_vals;
        uint32_t *r_head[2] = {d_head[0], d_head[1]};
        uint8_t *r_bwt = carry_bwt ? bwt_out : nullptr;
        uint8_t *r_hi = hi_out;
        uint64_t r_m = m, r_hw = hw;
        const uint32_t *r_diff = use_diff ? d_diff : nullptr;
        uint32_t *c_sa = nullptr, *c_orig = nullptr, *c_head[2] = {nullptr, nullptr};
        uint8_t *c_bw = nullptr, *c_hi = nullptr;
        uint64_t m_act = 0;
        const char *compact_env = std::getenv("DSMFM_REFINE_COMPACT"); // 0: refine in place (tests)
        const bool compact_off = compact_env && std::atoi(compact_env) == 0;
        const bool compact = use_diff && multi_step && !compact_off && remaining > 0;
        bool c_owned = false; // the dense arrays are allocations of their own (else: carved out of a key buffer)
        if (compact) {
            // scratch of the compaction: the key buffers of the initial sort are free from here on (the large-group
            // path, their only other user, starts later and never needs more than 8 bytes per dense entry)
            const uint64_t ntile = active_tiles(div_up(m, 32));
            uint32_t *d_act = reinterpret_cast<uint32_t *>(d_keys_a);
            uint64_t *d_tile = reinterpret_cast<uint64_t *>(d_keys_a) + (hw + 1) / 2;
            const bool scratch_fits = (hw + 1) / 2 + ntile + 1 <= m_max;
            if (!scratch_fits) {
                d_act = static_cast<uint32_t *>(dmalloc(hw * 4));
                d_tile = static_cast<uint64_t *>(dmalloc((ntile + 1) * 8));
            }
            DSM_CUDA(cudaMemsetAsync(d_act, 0, hw * 4, st));
            launch_mark_active(st, d_head[0], d_diff, m, d_act, d_tile, L);
            DSM_CUDA(cudaMemcpyAsync(&m_act, d_tile + ntile, 8, cudaMemcpyDeviceToHost, st));
            DSM_CUDA(cudaStreamSynchronize(st));
            stats.refine_members += m_act;
            if (m_act == 0) {
                remaining = 0; // every tie group carries a single BWT symbol
            } else if (m_act * 2 > remaining) {
                m_act = 0; // most members have to be sorted anyway (high repetition): refine in place
            } else {
                r_m = m_act;
                r_hw = head_words_for(m_act);
                auto up16 = [](uint64_t x) { return (x + 15) & ~(uint64_t)15; };
                const uint64_t b_sa = up16(m_act * 4 + 16), b_bw = up16(m_act + 16), b_hi = wide ? up16(m_act + 16) : 0,
                               b_head = up16(r_hw * 4);
                const uint64_t need = 2 * b_sa + b_bw + b_hi + 2 * b_head;
                // the upper part of the second key buffer, above what the large-group path can touch
                uint8_t *base = reinterpret_cast<uint8_t *>(d_keys_b) + up16(m_act * 8);
                c_owned = up16(m_act * 8) + need > m_max * 8;
                if (c_owned) base = static_cast<uint8_t *>(dmalloc(need));
                c_sa = reinterpret_cast<uint32_t *>(base);
                c_orig = reinterpret_cast<uint32_t *>(base + b_sa);
                c_bw = base + 2 * b_sa;
                c_hi = wide ? base + 2 * b_sa + b_bw : nullptr;
                c_head[0] = reinterpret_cast<uint32_t *>(base + 2 * b_sa + b_bw + b_hi);
                c_head[1] = reinterpret_cast<uint32_t *>(base + 2 * b_sa + b_bw + b_hi + b_head);
                DSM_CUDA(cudaMemsetAsync(c_head[0], 0, r_hw * 4, st));
                launch_compact_active(st, d_act, d_head[0], m, d_tile, d_sorted_vals, bwt_out, hi_out, m_act, c_sa, c_bw,
                                      c_hi, c_orig, c_head[0], r_hw, L);
                r_sa = c_sa;
                r_head[0] = c_head[0];
                r_head[1] = c_head[1];
                r_bwt = c_bw;
                r_hi = c_hi;
                r_diff = nullptr;
            }
            if (!scratch_fits) {
                dfree(d_act);
                dfree(d_tile);
            }
        } else if (remaining > 0) {
            stats.refine_members += remaining;
        }

        // ---- refinement rounds ------------------------------------------------------------
        // Suffixes that still agree on their first `depth` symbols are re-sorted by the next
        // SPW symbols taken straight from the packed text.  (The reference re-keys with the
        // ranks of the suffixes h positions ahead, utils.cpp:236-262; documents here are short,
        // the text fits in HBM next to the suffix array, and extending the key from the text
        // needs neither an inverse suffix array nor rank scatter traffic.)
        int cur = 0;
        uint32_t round = 0;
        uint32_t depth_next = (uint32_t)first_syms; // symbols every unresolved group is known to agree on
        const uint32_t max_rounds = (uint32_t)(maxgap / spw + 4);
        // windows that still own unresolved groups: all of them in the first round, a compact list afterwards
        const uint32_t nwin = (uint32_t)div_up(r_m, kRefWindow);
        const uint32_t *win_list = nullptr;
        uint32_t n_list = nwin;
        int wl = 0;
        while (remaining > 0) {
            if (round >= max_rounds)
                throw CudaError{cudaErrorUnknown, "refinement did not converge (internal error)", __FILE__, __LINE__};
            if (round < 32) stats.active[round] += remaining;
            ++round;
            const uint32_t depth = depth_next;
            DSM_CUDA(cudaMemcpyAsync(r_head[cur ^ 1], r_head[cur], r_hw * 4, cudaMemcpyDeviceToDevice, st));
            DSM_CUDA(cudaMemsetAsync(d_remaining, 0, 128 * 8, st));
            DSM_CUDA(cudaMemsetAsync(d_big_count, 0, 4, st));
            DSM_CUDA(cudaMemsetAsync(d_win_flag, 0, (size_t)nwin * 4, st));
            DSM_CUDA(cudaMemsetAsync(d_win_count, 0, 4, st));
            ++stats.refine_launches;
            launch_refine(st, bits, d_packed, r_sa, r_head[cur], r_head[cur ^ 1], r_m, depth, win_list, n_list,
                          d_big_heads, big_cap, d_big_count, d_remaining, d_win_flag, d_win_list[wl], d_win_count,
                          r_bwt, multi_step, key_words, r_hi, lo_bits, full_order, round == 1 ? r_diff : nullptr, L,
                          /*big_groups=*/!full_order && !(compact && m_act));
            uint32_t nbig = 0;
            DSM_CUDA(cudaMemcpyAsync(&nbig, d_big_count, 4, cudaMemcpyDeviceToHost, st));
            remaining = read_remaining();
            if (nbig > 0) {
                // groups too large for one CTA: one global (group, key) radix sort over all of them
                if (nbig > big_cap) throw CudaError{cudaErrorUnknown, "large-group list overflow", __FILE__, __LINE__};
                launch_big_extent(st, r_head[cur], r_m, d_big_heads, nbig, d_big_len, L);
                std::vector<uint32_t> heads(nbig), lens(nbig);
                DSM_CUDA(cudaMemcpyAsync(heads.data(), d_big_heads, (size_t)nbig * 4, cudaMemcpyDeviceToHost, st));
                DSM_CUDA(cudaMemcpyAsync(lens.data(), d_big_len, (size_t)nbig * 4, cudaMemcpyDeviceToHost, st));
                DSM_CUDA(cudaStreamSynchronize(st));
                std::vector<uint32_t> order(nbig);
                for (uint32_t i = 0; i < nbig; ++i) order[i] = i;
                std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return heads[a] < heads[b]; });
                std::vector<uint32_t> sheads(nbig);
                std::vector<uint64_t> offs(nbig + 1);
                uint64_t total = 0;
                for (uint32_t i = 0; i < nbig; ++i) {
                    sheads[i] = heads[order[i]];
                    offs[i] = total;
                    total += lens[order[i]];
                }
                offs[nbig] = total;
                stats.fallback_elems += total;
                uint64_t *d_off = static_cast<uint64_t *>(dmalloc((size_t)(nbig + 1) * 8));
                uint32_t *d_bsa = static_cast<uint32_t *>(dmalloc(total * 4));
                uint32_t *d_bgid = static_cast<uint32_t *>(dmalloc(total * 4));
                uint64_t *d_bkey = static_cast<uint64_t *>(dmalloc(total * 8));
                uint32_t *d_perm = static_cast<uint32_t *>(dmalloc(total * 4 + 16));
                uint8_t *d_bhi = wide ? static_cast<uint8_t *>(dmalloc(total + 16)) : nullptr;
                DSM_CUDA(cudaMemcpyAsync(d_big_heads, sheads.data(), (size_t)nbig * 4, cudaMemcpyHostToDevice, st));
                DSM_CUDA(cudaMemcpyAsync(d_off, offs.data(), (size_t)(nbig + 1) * 8, cudaMemcpyHostToDevice, st));
                launch_big_gather(st, bits, d_packed, r_sa, depth, d_big_heads, d_off, nbig, total, d_bsa,
                                  d_bkey, d_bgid, r_hi, d_bhi, lo_bits, L);
                // the key buffers of the initial sort are free by now
                DSM_CUDA(cudaMemcpyAsync(d_keys_a, d_bkey, total * 8, cudaMemcpyDeviceToDevice, st));
                int p1 = radix_sort_pairs(st, ws, d_keys_a, d_other_vals, d_keys_b, d_perm, total, 0, full_key_bits, true, L);
                // pass 0 writes (keys_b, perm); an odd pass count leaves the result there
                uint64_t *kfree = (p1 & 1) ? d_keys_a : d_keys_b;
                uint32_t *pres = (p1 & 1) ? d_perm : d_other_vals;
                uint32_t *pfree = (p1 & 1) ? d_other_vals : d_perm;
                if (nbig > 1) {
                    int gbits = 1;
                    while ((1ull << gbits) < nbig) ++gbits;
                    launch_gather_u32_to_u64(st, d_bgid, pres, total, kfree, L);
                    uint64_t *k2a = kfree, *k2b = (kfree == d_keys_a) ? d_keys_b : d_keys_a;
                    int p2 = radix_sort_pairs(st, ws, k2a, pres, k2b, pfree, total, 0, gbits, false, L);
                    if (p2 & 1) std::swap(pres, pfree);
                }
                launch_big_scatter(st, bits, pres, d_bsa, d_bkey, d_bgid, d_big_heads, d_off, total, r_sa,
                                   r_head[cur ^ 1], d_win_flag, d_win_list[wl], d_win_count, d_packed, d_inv,
                                   r_bwt, d_bhi, r_hi, lo_bits, L);
                DSM_CUDA(cudaStreamSynchronize(st)); // sheads / offs are host vectors
                dfree(d_off);
                dfree(d_bsa);
                dfree(d_bgid);
                dfree(d_bkey);
                dfree(d_perm);
                dfree(d_bhi);
                remaining += total; // re-examined (and counted exactly) by the next round
            }
            // a CTA step consumes key_words*SPW symbols, the large-group path SPW; starting the next launch at the
            // smaller of the two is always safe (already-equal symbols just compare equal again)
            depth_next = depth + ((multi_step || nbig > 0) ? (uint32_t)spw : (uint32_t)(key_words * spw));
            DSM_CUDA(cudaMemcpyAsync(&n_list, d_win_count, 4, cudaMemcpyDeviceToHost, st));
            DSM_CUDA(cudaStreamSynchronize(st));
            win_list = d_win_list[wl];
            wl ^= 1;
            cur ^= 1;
            if (remaining > 0 && n_list == 0)
                throw CudaError{cudaErrorUnknown, "unresolved groups without an owning window (internal error)", __FILE__, __LINE__};
        }
        if (compact && m_act) { // the BWT bytes of the sorted groups go back to their slots
            launch_scatter_bwt(st, c_orig, c_bw, m_act, bwt_out, L);
            if (c_owned) dfree(c_sa);
        }
        rounds_max = std::max(rounds_max, round);
        // ---- BWT when it could not ride along (64-bit first keys, unsharded only) -----------
        if (!carry_bwt) launch_bwt(st, bits, d_packed, d_inv, d_sorted_vals, m, bwt_out, L);
        if (d_sa_all) DSM_CUDA(cudaMemcpyAsync(d_sa_all + off, d_sorted_vals, m * 4, cudaMemcpyDeviceToDevice, st));
        DSM_CUDA(cudaEventRecord(evr[2], st));
        DSM_CUDA(cudaStreamSynchronize(st));
        trace("build: refinement done");
        float ms;
        cudaEventElapsedTime(&ms, evr[0], evr[1]); ms_sort += ms;
        cudaEventElapsedTime(&ms, evr[1], evr[2]); ms_refine += ms;
        if (passes) { cudaEventElapsedTime(&ms, ev_pass0, ev_pass1); ms_passes += ms; }
        off += m;
    }
    for (auto &e : evr) cudaEventDestroy(e);
    dfree(d_win_flag);
    dfree(d_win_list[0]);
    dfree(d_win_list[1]);
    dfree(d_win_count);
    stats.rounds = rounds_max;
    stats.sort_pass_bytes = pass_launches ? pass_launch_bytes / pass_launches : 0;
    stats.sort_launches = pass_launches;
    DSM_CUDA(cudaEventRecord(ev[3], st));
    DSM_CUDA(cudaEventRecord(ev[4], st));

    // ---- C table, code table, wavelet tree ---------------------------------------------
    index.C[0] = 0;
    for (int i = 1; i < 256; ++i) index.C[i] = index.C[i - 1] + counts[i - 1]; // FMIndex.cpp:397-409
    const uint32_t maxbits = build_codetable(counts, index.codetable);
    if (maxbits > 32)
        throw CudaError{cudaErrorInvalidValue, "Huffman code longer than 32 bits (the .fmi code field holds 32)", __FILE__, __LINE__};
    if (!sharded) {
        size_t wt_bytes = 0;
        wavelet_build_device(st, d_bwt, n, index.codetable, wt, L, &wt_bytes);
        dev_now += wt_bytes;
        dev_peak = std::max(dev_peak, dev_now);
        dev_now -= wt_bytes - std::min(wt_bytes, wt.section_bytes);
    }
    DSM_CUDA(cudaEventRecord(ev[5], st));
    DSM_CUDA(cudaStreamSynchronize(st));
    trace("build: wavelet tree done");

    // ---- release what the sections do not need ---------------------------------------
    pipeline_drop_spec(); // (d_hist, d_map of a streamed batch)
    dfree(d_map);
    dfree(d_inv);
    dfree(d_sel_lut);
    if (!packed_in) dfree(d_packed);
    dfree(d_keys_a);
    dfree(d_keys_b);
    dfree(d_head[0]);
    dfree(d_head[1]);
    dfree(d_diff);
    dfree(d_remaining);
    dfree(d_big_heads);
    dfree(d_big_len);
    dfree(d_big_count);
    dfree(ws.hist);
    dfree(ws.carry);
    dfree(ws.status);
    dfree(ws.counter);
    dfree(d_last_other_vals);
    if (sharded) {
        dfree(d_last_sorted_vals);
        d_sa = d_sa_all;
        if (keep_sa) d_sa_hi = d_hi_buf; else dfree(d_hi_buf);
    } else if (keep_sa) {
        d_sa = d_last_sorted_vals;
    } else {
        dfree(d_last_sorted_vals);
    }
    pos_lo_bits = lo_bits;
    if (packed_in && keep_sa) sa_derive(bits, L);

    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[5]); stats.ms_total = ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); stats.ms_pack = ms;
    stats.ms_sort = ms_sort;
    stats.ms_sort_pass = pass_launches ? ms_passes / pass_launches : 0.f;
    stats.ms_refine = ms_refine;
    stats.ms_bwt = 0.f; // the BWT rides through the sort (or is gathered inside the range loop)
    cudaEventElapsedTime(&ms, ev[4], ev[5]); stats.ms_wt = ms;
    stats.device_bytes_peak = dev_peak;
    for (auto &e : ev) cudaEventDestroy(e);
    cudaEventDestroy(ev_pass0);
    cudaEventDestroy(ev_pass1);
    stats.kernel_launches += pre_launches;
    built = true;
}

void dsmfm_builder::fetch()
{
    cudaEvent_t e0, e1;
    DSM_CUDA(cudaEventCreate(&e0));
    DSM_CUDA(cudaEventCreate(&e1));
    trace("fetch: begin");
    DSM_CUDA(cudaEventRecord(e0, stream));
    uint8_t *ready = nullptr;
    if (host_prefetch.joinable()) {
        host_prefetch.join();
        if (host_ready_bytes >= wt.section_bytes && wt.shape.n_internal > 0) ready = host_ready;
        else g_pinned.put(host_ready);
        host_ready = nullptr;
    }
    wavelet_fetch(stream, wt, ready);
    trace("fetch: sections in host memory");
    if ((flags & DSMFM_FLAG_KEEP_BWT) && shard_count <= 1) {
        h_bwt = static_cast<uint8_t *>(g_pinned.get(index.n));
        DSM_CUDA(cudaMemcpyAsync(h_bwt, d_bwt, index.n, cudaMemcpyDeviceToHost, stream));
    }
    DSM_CUDA(cudaEventRecord(e1, stream));
    DSM_CUDA(cudaStreamSynchronize(stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    stats.ms_d2h = ms;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    index.n_nodes = (uint32_t)wt.shape.nodes.size();
    index.nodes = wt.shape.nodes.data();
    index.bwt = h_bwt;
    // the device copies are no longer needed (the .sa writer still wants the BWT)
    if (!(flags & DSMFM_FLAG_KEEP_SA)) {
        dfree(d_bwt);
        d_bwt = nullptr;
    }
    dev_free(wt.d_sections, stream);
    dev_free(wt.d_ch, stream);
    wt.d_sections = wt.d_ch = nullptr;
    fetched = true;
}

// ---------------------------------------------------------------------------
// .sa image: FMIndex::saveSamples over maketables (FMIndex.cpp:125-147, 572-714).  The reference
// walks the whole text backwards by LF-mapping to find the sampled BWT positions and the order of
// the end markers; with the suffix array in HBM the same tables fall out of three passes over it.
// ---------------------------------------------------------------------------
namespace {
unsigned ceil_log2(uint64_t i) // Tools::CeilLog2, Tools.cpp:43-64
{
    unsigned b = 0;
    uint64_t t = i;
    while (t) { ++b; t >>= 1; }
    const unsigned fl = b ? b - 1 : 0;
    return ((uint64_t)1 << fl) != i ? fl + 1 : fl;
}

// BlockArray::Save (BlockArray.h:54-64): n, blockLength, n*blockLength/64+1 words, fields LSB first (Tools.h:49-61)
void put_block_array(std::vector<uint8_t> &out, const uint32_t *v, uint64_t count, unsigned len)
{
    std::vector<uint64_t> data(count * len / 64 + 1, 0);
    if (len)
        for (uint64_t i = 0; i < count; ++i) {
            const uint64_t bit = i * len, w = bit >> 6, j = bit & 63, x = v[i];
            data[w] |= x << j;
            if (j + len > 64) data[w + 1] |= x >> (64 - j);
        }
    const uint64_t hdr[2] = {count, len};
    const uint8_t *h = reinterpret_cast<const uint8_t *>(hdr), *d = reinterpret_cast<const uint8_t *>(data.data());
    out.insert(out.end(), h, h + 16);
    out.insert(out.end(), d, d + data.size() * 8);
}
} // namespace

void dsmfm_builder::make_sa_image()
{
    cudaStream_t st = stream;
    uint32_t *L = &stats.kernel_launches;
    const uint64_t nn = index.n;
    const uint32_t D = index.number_of_texts;
    const uint64_t words = nn / 64 + 1, nsb = nn / 256 + 1, nb = nn / 64 + 1;
    struct Bits {
        uint64_t *data = nullptr, *Rs = nullptr;
        uint8_t *Rb = nullptr;
    };
    uint32_t *d_mark = static_cast<uint32_t *>(dmalloc(((nn >> 5) + 2) * 4));
    uint64_t *d_scratch = static_cast<uint64_t *>(dmalloc(sizeof(uint64_t) * (div_up(nsb, kRankChunk) + 1)));
    Bits sampled, starts;
    for (Bits *b : {&sampled, &starts}) {
        b->data = static_cast<uint64_t *>(dmalloc(words * 8));
        b->Rs = static_cast<uint64_t *>(dmalloc(nsb * 8));
        b->Rb = static_cast<uint8_t *>(dmalloc(nb + 8));
    }
    DSM_CUDA(cudaMemsetAsync(d_mark, 0, ((nn >> 5) + 2) * 4, st));
    launch_sa_mark(st, d_doc_end, D, samplerate, d_mark, L);
    launch_sa_rank_bits(st, d_sa, nullptr, d_mark, nn, reinterpret_cast<uint32_t *>(sampled.data), words * 2, L);
    launch_bitrank(st, sampled.data, nn, sampled.Rs, sampled.Rb, d_scratch, L);
    launch_sa_rank_bits(st, d_sa, d_bwt, nullptr, nn, reinterpret_cast<uint32_t *>(starts.data), words * 2, L);
    launch_bitrank(st, starts.data, nn, starts.Rs, starts.Rb, d_scratch, L);

    std::vector<uint64_t> h_data(words), h_rs(nsb);
    std::vector<uint8_t> h_rb(nb);
    DSM_CUDA(cudaMemcpyAsync(h_data.data(), sampled.data, words * 8, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(h_rs.data(), sampled.Rs, nsb * 8, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(h_rb.data(), sampled.Rb, nb, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    uint64_t samples = h_rs[nsb - 1];
    for (uint64_t w = 4 * (nsb - 1); w < words; ++w) samples += (uint64_t)__builtin_popcountll(h_data[w]);

    uint32_t *d_sdoc = static_cast<uint32_t *>(dmalloc(samples * 4 + 16));
    uint32_t *d_soff = static_cast<uint32_t *>(dmalloc(samples * 4 + 16));
    uint32_t *d_emdoc = static_cast<uint32_t *>(dmalloc((size_t)D * 4 + 16));
    launch_sa_emit(st, d_sa, sampled.data, sampled.Rs, sampled.Rb, nn, d_doc_end, D, d_sdoc, d_soff, L);
    launch_sa_emit(st, d_sa, starts.data, starts.Rs, starts.Rb, nn, d_doc_end, D, d_emdoc, nullptr, L);
    std::vector<uint32_t> h_sdoc(samples + 1), h_soff(samples + 1), h_emdoc(D), h_end(D), h_len(D);
    DSM_CUDA(cudaMemcpyAsync(h_sdoc.data(), d_sdoc, samples * 4, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(h_soff.data(), d_soff, samples * 4, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(h_emdoc.data(), d_emdoc, (size_t)D * 4, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaMemcpyAsync(h_end.data(), d_doc_end, (size_t)D * 4, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    dfree(d_mark); dfree(d_scratch); dfree(d_sdoc); dfree(d_soff); dfree(d_emdoc);
    for (Bits *b : {&sampled, &starts}) { dfree(b->data); dfree(b->Rs); dfree(b->Rb); }
    for (uint32_t k = 0; k < D; ++k) h_len[k] = h_end[k] - (k ? h_end[k - 1] + 1 : 0u); // FMIndex.cpp:703-707

    // saveSamples order: sampled (BitRank::save), suffixes, suffixDocId, textLength, Doc (FMIndex.cpp:134-143)
    std::vector<uint8_t> &out = sa_image;
    out.clear();
    const uint64_t integers = (nn + 1) % 64 ? (nn + 1) / 64 + 1 : (nn + 1) / 64;
    const uint32_t b64 = 64, s256 = 256;
    auto put = [&](const void *p, size_t bytes) {
        const uint8_t *q = static_cast<const uint8_t *>(p);
        out.insert(out.end(), q, q + bytes);
    };
    put(&nn, 8); put(&integers, 8); put(&b64, 4); put(&s256, 4);
    put(h_data.data(), integers * 8); put(h_rs.data(), nsb * 8); put(h_rb.data(), nb);
    const unsigned wlen = ceil_log2(index.max_text_length), wdoc = ceil_log2(D);
    put_block_array(out, h_soff.data(), samples, wlen);
    put_block_array(out, h_sdoc.data(), samples, wdoc);
    put_block_array(out, h_len.data(), D, wlen);
    put_block_array(out, h_emdoc.data(), D, wdoc);
}

// .sa samples of a packed-text build: what needs the replicated text or the slice's BWT is derived here, before the
// caller releases the text (right after dsmfm_build_packed) and dsmfm_pieces_build the BWT.  Positions are positions
// in the padded text; the document of a position and its offset follow from the document ends alone.
void dsmfm_builder::sa_derive(int bits, uint32_t *L)
{
    cudaStream_t st = stream;
    const uint64_t spw = 64 / (uint64_t)bits, n_text = ext->words * spw, D = counts[0];
    sah = SaHost();
    sah.slot_syms = ext->geom.slot_words * spw;
    sah.world = ext->geom.world;
    sah.d_doc_end = static_cast<uint64_t *>(dmalloc(D * 8 + 16));
    uint64_t *d_tile = static_cast<uint64_t *>(dmalloc(term_tiles(n_text) * 8));
    launch_packed_term_positions(st, bits, ext->text, n_text, ext->geom, d_tile, sah.d_doc_end, L);
    dfree(d_tile);
    const size_t mark_bytes = (n_text / 32 + 2) * 4;
    uint32_t *d_mark = static_cast<uint32_t *>(dmalloc(mark_bytes));
    DSM_CUDA(cudaMemsetAsync(d_mark, 0, mark_bytes, st));
    launch_sa_mark64(st, sah.d_doc_end, (uint32_t)D, samplerate, sah.slot_syms, d_mark, L);
    size_t blob = 0;
    const VecPiece l = vec_layout(shard_rank_begin, shard_m, index.n, false, true, blob);
    const size_t ends_bytes = (shard_m / 64 + 1) * 8;
    sah.d_sampled = static_cast<uint64_t *>(dmalloc(l.words * 8));
    sah.d_ends = static_cast<uint64_t *>(dmalloc(ends_bytes));
    unsigned long long *d_cnt = static_cast<unsigned long long *>(dmalloc(16));
    DSM_CUDA(cudaMemsetAsync(sah.d_sampled, 0, l.words * 8, st));
    DSM_CUDA(cudaMemsetAsync(sah.d_ends, 0, ends_bytes, st));
    DSM_CUDA(cudaMemsetAsync(d_cnt, 0, 16, st));
    launch_sa_slice_bits(st, d_sa, d_sa_hi, pos_lo_bits, d_bwt, d_mark, shard_m, sah.d_sampled, l.base, sah.d_ends, d_cnt, L);
    unsigned long long cnt[2] = {0, 0};
    DSM_CUDA(cudaMemcpyAsync(cnt, d_cnt, sizeof cnt, cudaMemcpyDeviceToHost, st));
    DSM_CUDA(cudaStreamSynchronize(st));
    dfree(d_mark);
    dfree(d_cnt);
    sah.info.samples = cnt[0];
    sah.info.ends = cnt[1];
    sah.info.documents = block_info.documents;
    sah.ready = true;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
#define API_GUARD(b)                                             \
    if (!(b)) return DSMFM_EINVAL;                                \
    cudaSetDevice((b)->device)

extern "C" {

DSMFM_API int dsmfm_version(void) { return DSMFM_VERSION; }

DSMFM_API int dsmfm_create(const dsmfm_options *opts, dsmfm_builder **out)
{
    if (!out) return DSMFM_EINVAL;
    *out = nullptr;
    trace("dsmfm_create");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device available: ") + cudaGetErrorString(e) +
                         " (this library has no CPU fallback)";
        return DSMFM_ECUDA;
    }
    int dev = opts ? opts->device : -1;
    if (dev < 0) cudaGetDevice(&dev);
    if (dev >= ndev) {
        g_create_error = "device ordinal out of range";
        return DSMFM_EINVAL;
    }
    int cc_major = 0; // (cudaGetDeviceProperties takes tens of milliseconds; one attribute does not)
    if ((e = cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev)) != cudaSuccess || cc_major < 10) {
        g_create_error = "device is not sm_100 or newer (kernels are built for sm_100a only)";
        return DSMFM_ECUDA;
    }
    dsmfm_builder *b = new (std::nothrow) dsmfm_builder();
    if (!b) return DSMFM_ENOMEM;
    b->device = dev;
    std::memset(&b->index, 0, sizeof b->index);
    std::memset(&b->stats, 0, sizeof b->stats);
    std::memset(b->counts, 0, sizeof b->counts);
    if (opts) {
        b->samplerate = opts->samplerate ? opts->samplerate : DSMFM_DEFAULT_SAMPLERATE;
        b->flags = opts->flags;
        b->expected = opts->expected_bytes;
        b->stream = static_cast<cudaStream_t>(opts->stream);
        b->shard_count = opts->shard_count ? opts->shard_count : 1;
        b->shard_index = opts->shard_index;
        b->shard_span = opts->shard_span ? opts->shard_span : 1;
        if (b->shard_index >= b->shard_count || b->shard_span > b->shard_count - b->shard_index) {
            g_create_error = "shard_index / shard_span out of range";
            delete b;
            return DSMFM_EINVAL;
        }
    }
    try {
        DSM_CUDA(cudaSetDevice(dev));
        {
            // keep freed device memory in the pool between builds (see dev_alloc)
            cudaMemPool_t pool;
            DSM_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
            uint64_t keep = ~0ull;
            DSM_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        }
        // opts->stream == NULL means "a stream of the builder's own" unless the caller states that it really
        // wants the legacy default stream (handle 0), e.g. because its own work is queued there
        if (!b->stream && !(b->flags & DSMFM_FLAG_DEFAULT_STREAM)) {
            DSM_CUDA(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
            b->own_stream = true;
        }
    } catch (const CudaError &ce) {
        g_create_error = std::string("CUDA error: ") + cudaGetErrorString(ce.code);
        delete b;
        return DSMFM_ECUDA;
    }
    trace("dsmfm_create: device, pool and stream ready");
    *out = b;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_append(dsmfm_builder *b, const uint8_t *doc, size_t len)
{
    API_GUARD(b);
    if (b->finished || b->sealed) return b->fail(DSMFM_EINVAL, "dsmfm_append: new text can not be inserted after dsmfm_finish");
    if (!doc) return b->fail(DSMFM_EINVAL, "dsmfm_append: null document");
    if (len == 0) return b->fail(DSMFM_EEMPTY, "dsmfm_append: can not index empty texts");
    try {
        if (!b->stage[0]) {
            for (int i = 0; i < 2; ++i) {
                b->stage[i] = static_cast<uint8_t *>(g_pinned.get(dsmfm_builder::kStage));
                DSM_CUDA(cudaEventCreateWithFlags(&b->stage_free[i], cudaEventDisableTiming));
            }
        }
        const uint8_t *p = doc;
        size_t left = len;
        while (left) { // documents longer than the staging buffer are split across flushes
            if (b->cur_used == dsmfm_builder::kStage) b->flush_stage();
            const size_t take = std::min(left, dsmfm_builder::kStage - b->cur_used);
            std::memcpy(b->stage[b->cur] + b->cur_used, p, take);
            b->cur_used += take;
            p += take;
            left -= take;
        }
        if (b->cur_used == dsmfm_builder::kStage) b->flush_stage();
        b->stage[b->cur][b->cur_used++] = 0;
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

static int append_bulk(dsmfm_builder *b, const void *src, size_t bytes, cudaMemcpyKind kind)
{
    if (b->finished || b->sealed) return b->fail(DSMFM_EINVAL, "append: new text can not be inserted after dsmfm_finish");
    if (!src || bytes == 0) return b->fail(DSMFM_EINVAL, "append: empty batch");
    try {
        b->flush_stage();
        b->pipeline_abandon(); // (a second batch behind a streamed one: plain statistics at build time)
        if (kind != cudaMemcpyHostToDevice || !b->append_pipelined(static_cast<const uint8_t *>(src), bytes))
            b->push_device(src, bytes, kind);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_append_batch(dsmfm_builder *b, const uint8_t *docs, size_t bytes)
{
    API_GUARD(b);
    if (docs && bytes && docs[bytes - 1] != 0)
        return b->fail(DSMFM_EINVAL, "dsmfm_append_batch: the batch must end with a document terminator");
    return append_bulk(b, docs, bytes, cudaMemcpyHostToDevice);
}

DSMFM_API int dsmfm_append_batch_device(dsmfm_builder *b, const void *docs_dev, size_t bytes)
{
    API_GUARD(b);
    return append_bulk(b, docs_dev, bytes, cudaMemcpyDeviceToDevice);
}

DSMFM_API int dsmfm_append_fasta(dsmfm_builder *b, const uint8_t *text, size_t len, int final, dsmfm_fasta_info *info)
{
    API_GUARD(b);
    if (!info) return b->fail(DSMFM_EINVAL, "dsmfm_append_fasta: null info");
    std::memset(info, 0, sizeof *info);
    info->first_invalid_offset = ~0ull;
    if (b->finished || b->sealed) return b->fail(DSMFM_EINVAL, "dsmfm_append_fasta: new text can not be inserted after dsmfm_finish");
    if (!text && len) return b->fail(DSMFM_EINVAL, "dsmfm_append_fasta: null text");
    size_t use = 0;
    if (final) {
        // `getline(...).good()`: a last line without '\n' is dropped (builder.cpp:211)
        const void *p = len ? memrchr(text, '\n', len) : nullptr;
        use = p ? (size_t)(static_cast<const uint8_t *>(p) - text) + 1 : 0;
        info->consumed = len;
    } else {
        // everything in front of the last header line: the record it opens may continue in the next call
        size_t i = len;
        while (i > 0) {
            const void *p = memrchr(text, '>', i);
            if (!p) break;
            const size_t q = (size_t)(static_cast<const uint8_t *>(p) - text);
            if (q == 0 || text[q - 1] == '\n') {
                use = q;
                break;
            }
            i = q;
        }
        info->consumed = use;
    }
    if (use == 0) return DSMFM_OK;
    try {
        b->flush_stage();
        b->append_fasta(text, use, info);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API void *dsmfm_alloc_pinned(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

DSMFM_API void dsmfm_free_pinned(void *p)
{
    if (p) cudaFreeHost(p);
}

static int run_build(dsmfm_builder *b)
{
    b->finished = true;
    const double t0 = now_ms();
    g_alloc_ms = 0.0;
    try {
        b->build();
        b->stats.ms_wall_build = (float)(now_ms() - t0);
        b->stats.ms_wall_alloc = (float)g_alloc_ms;
    } catch (const CudaError &e) {
        b->release_device();
        if (e.what && std::strcmp(e.what, "EMPTY") == 0)
            return b->fail(DSMFM_EEMPTY, "can not index empty texts (two consecutive terminators in the input)");
        if (e.code == cudaErrorInvalidValue && e.what && std::strstr(e.what, "2^32"))
            return b->fail(DSMFM_ELIMIT, "%s", e.what);
        if (e.code == cudaErrorInvalidValue && e.what && std::strstr(e.what, "Huffman"))
            return b->fail(DSMFM_ELIMIT, "%s", e.what);
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        b->release_device();
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_build_device(dsmfm_builder *b)
{
    API_GUARD(b);
    if (b->finished) return b->fail(DSMFM_EINVAL, "dsmfm_build_device: already built");
    if (b->sealed) return b->fail(DSMFM_EINVAL, "dsmfm_build_device: the block belongs to a packed-text build (dsmfm_build_packed)");
    return run_build(b);
}

// ---- one collection over several builders: packed-text exchange ---------------------------------

DSMFM_API int dsmfm_block_stats(dsmfm_builder *b, dsmfm_block_info *out)
{
    API_GUARD(b);
    if (!out) return DSMFM_EINVAL;
    if (b->finished) return b->fail(DSMFM_EINVAL, "dsmfm_block_stats: already built");
    try {
        b->flush_stage();
        if (b->pl.active) { // a streamed batch: statistics are ready; its pack used the LOCAL alphabet and is dropped
            b->pipeline_finish_stats();
            b->pipeline_drop_spec();
        }
        if (b->n == 0) {
            std::memset(&b->block_info, 0, sizeof b->block_info);
            b->block_stats_done = true;
        } else {
            b->gather_raw();
            if (!b->block_stats_done) b->block_stats(&b->pre_launches);
        }
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    b->sealed = true;
    *out = b->block_info;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_text_plan_make(const dsmfm_block_info *all, uint32_t world, dsmfm_text_plan *out)
{
    if (!all || !out || world == 0 || world > DSMFM_MAX_BLOCKS) return DSMFM_EINVAL;
    std::memset(out, 0, sizeof *out);
    out->world = world;
    for (uint32_t r = 0; r < world; ++r) {
        if (all[r].empty_document) return DSMFM_EEMPTY;
        for (int c = 0; c < 256; ++c) out->counts[c] += all[r].counts[c];
        out->n += all[r].bytes;
        out->documents += all[r].documents;
        out->max_text_length = std::max(out->max_text_length, all[r].max_text_length);
        out->block_bytes[r] = all[r].bytes;
    }
    uint32_t sigma = 0;
    for (int c = 1; c < 256; ++c) sigma += out->counts[c] != 0;
    out->bits = sigma <= 7 ? 3 : (sigma <= 15 ? 4 : 8);
    const uint64_t spw = 64 / out->bits;
    uint64_t slot = 1;
    for (uint32_t r = 0; r < world; ++r) slot = std::max(slot, div_up(all[r].bytes, spw));
    out->slot_words = (slot + 15) & ~(uint64_t)15; // whole 128-byte lines per slot
    out->text_bytes = (out->slot_words * world + 8) * 8;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_block_pack(dsmfm_builder *b, const dsmfm_text_plan *plan, uint32_t rank, void *text_dev,
                               uint64_t *top_hist4096)
{
    API_GUARD(b);
    if (!plan || !text_dev || !top_hist4096 || rank >= plan->world || plan->world > DSMFM_MAX_BLOCKS)
        return b->fail(DSMFM_EINVAL, "dsmfm_block_pack: bad arguments");
    if (!b->sealed || b->finished) return b->fail(DSMFM_EINVAL, "dsmfm_block_pack: call dsmfm_block_stats first");
    if (plan->block_bytes[rank] != b->n) return b->fail(DSMFM_EINVAL, "dsmfm_block_pack: block %u of the plan is not this builder's", rank);
    try {
        cudaStream_t st = b->stream;
        uint32_t *L = &b->pre_launches;
        uint8_t code_map[256];
        std::memset(code_map, 0, sizeof code_map);
        uint32_t sigma = 0;
        for (int c = 1; c < 256; ++c)
            if (plan->counts[c]) code_map[c] = (uint8_t)++sigma;
        const int bits = (int)plan->bits, spw = 64 / bits;
        uint64_t *slot = static_cast<uint64_t *>(text_dev) + (uint64_t)rank * plan->slot_words;
        uint8_t *d_map = static_cast<uint8_t *>(b->dmalloc(256));
        unsigned long long *d_top = static_cast<unsigned long long *>(b->dmalloc(4096 * 8));
        DSM_CUDA(cudaMemcpyAsync(d_map, code_map, 256, cudaMemcpyHostToDevice, st));
        DSM_CUDA(cudaMemsetAsync(d_top, 0, 4096 * 8, st));
        // the slot: the block's symbols, then zeros; 8 zero words behind the last slot of this device's copy
        launch_pack(st, bits, b->d_raw, b->n, d_map, slot, plan->slot_words, L);
        DSM_CUDA(cudaMemsetAsync(static_cast<uint64_t *>(text_dev) + (uint64_t)plan->world * plan->slot_words, 0, 64, st));
        if (b->n) launch_key_top_hist(st, bits, slot, b->n, spw, 12, d_top, L);
        static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "histogram words");
        DSM_CUDA(cudaMemcpyAsync(top_hist4096, d_top, 4096 * 8, cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaStreamSynchronize(st));
        b->dfree(d_map);
        b->dfree(d_top);
        if (b->d_raw) b->dfree(b->d_raw);
        b->chunks.clear();
        b->d_raw = nullptr;
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_build_packed(dsmfm_builder *b, const dsmfm_text_plan *plan, const void *text_dev,
                                 const uint64_t *top_hist4096)
{
    API_GUARD(b);
    if (!plan || !text_dev || !top_hist4096 || plan->world == 0 || plan->world > DSMFM_MAX_BLOCKS)
        return b->fail(DSMFM_EINVAL, "dsmfm_build_packed: bad arguments");
    if (b->finished) return b->fail(DSMFM_EINVAL, "dsmfm_build_packed: already built");
    if (!b->sealed || b->d_raw) return b->fail(DSMFM_EINVAL, "dsmfm_build_packed: call dsmfm_block_stats and dsmfm_block_pack first");
    if ((b->flags & DSMFM_FLAG_KEEP_SA) && plan->documents >= (1ull << 32))
        return b->fail(DSMFM_ELIMIT, "dsmfm_build_packed: .sa samples of 2^32 documents or more (document ids are u32)");
    if (plan->n == 0) return b->fail(DSMFM_EINVAL, "dsmfm_build_packed: empty collection (build it with dsmfm_finish on one builder)");
    uint64_t total = 0;
    for (int i = 0; i < 4096; ++i) total += top_hist4096[i];
    if (total != plan->n) return b->fail(DSMFM_EINVAL, "dsmfm_build_packed: the key histogram does not add up to the collection");
    auto *ext = new (std::nothrow) dsmfm_builder::PackedText();
    if (!ext) return b->fail(DSMFM_ENOMEM, "host allocation failed");
    ext->text = static_cast<const uint64_t *>(text_dev);
    std::memset(&ext->geom, 0, sizeof ext->geom);
    ext->geom.slot_words = plan->slot_words;
    ext->geom.world = plan->world;
    for (uint32_t r = 0; r < plan->world; ++r) ext->geom.bytes[r] = plan->block_bytes[r];
    ext->n_real = plan->n;
    ext->words = plan->slot_words * plan->world;
    ext->documents = plan->documents;
    ext->maxlen = plan->max_text_length;
    ext->top.assign(top_hist4096, top_hist4096 + 4096);
    delete b->ext;
    b->ext = ext;
    std::memcpy(b->counts, plan->counts, sizeof b->counts);
    return run_build(b);
}

DSMFM_API int dsmfm_shard_info(dsmfm_builder *b, dsmfm_shard *out)
{
    API_GUARD(b);
    if (!out) return DSMFM_EINVAL;
    if (!b->built) return b->fail(DSMFM_EINVAL, "dsmfm_shard_info: nothing built");
    out->n_total = b->index.n;
    out->rank_begin = b->shard_rank_begin;
    out->count = b->shard_m;
    out->bwt_dev = b->d_bwt;
    out->sa_dev = nullptr;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_shard_export(dsmfm_builder *b, void *bwt_dst_dev, void *sa_dst_dev)
{
    API_GUARD(b);
    if (!b->built || !b->d_bwt) return b->fail(DSMFM_EINVAL, "dsmfm_shard_export: nothing built (or already fetched)");
    if (sa_dst_dev && !b->d_sa) return b->fail(DSMFM_EINVAL, "dsmfm_shard_export: the suffix array needs DSMFM_FLAG_KEEP_SA");
    const uint64_t m = b->shard_count > 1 ? b->shard_m : b->index.n;
    try {
        if (bwt_dst_dev && m) DSM_CUDA(cudaMemcpyAsync(bwt_dst_dev, b->d_bwt, m, cudaMemcpyDeviceToDevice, b->stream));
        if (sa_dst_dev)
            launch_widen_sa(b->stream, b->d_sa, b->d_sa_hi, b->pos_lo_bits, m, static_cast<uint64_t *>(sa_dst_dev),
                            &b->stats.kernel_launches);
        DSM_CUDA(cudaStreamSynchronize(b->stream));
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_assemble(dsmfm_builder *b, const void *bwt_dev, uint64_t n_total)
{
    API_GUARD(b);
    if (!b->built || b->shard_count <= 1) return b->fail(DSMFM_EINVAL, "dsmfm_assemble: needs a built sharded builder");
    if (b->assembled) return b->fail(DSMFM_EINVAL, "dsmfm_assemble: already assembled");
    if (!bwt_dev || n_total != b->index.n) return b->fail(DSMFM_EINVAL, "dsmfm_assemble: BWT size does not match the collection");
    try {
        cudaEvent_t e0, e1;
        DSM_CUDA(cudaEventCreate(&e0));
        DSM_CUDA(cudaEventCreate(&e1));
        DSM_CUDA(cudaEventRecord(e0, b->stream));
        wavelet_build_device(b->stream, static_cast<const uint8_t *>(bwt_dev), n_total, b->index.codetable, b->wt,
                             &b->stats.kernel_launches, nullptr);
        DSM_CUDA(cudaEventRecord(e1, b->stream));
        DSM_CUDA(cudaStreamSynchronize(b->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        b->stats.ms_wt = ms;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    b->assembled = true;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_slice_hist(dsmfm_builder *b, uint64_t *out256)
{
    API_GUARD(b);
    if (!out256) return DSMFM_EINVAL;
    if (!b->built || !b->d_bwt) return b->fail(DSMFM_EINVAL, "dsmfm_slice_hist: nothing built (or already fetched)");
    const uint64_t m = b->shard_count > 1 ? b->shard_m : b->index.n;
    try {
        uint64_t *d_counts = static_cast<uint64_t *>(dev_alloc(256 * 8, b->stream));
        DSM_CUDA(cudaMemsetAsync(d_counts, 0, 256 * 8, b->stream));
        if (m) launch_byte_hist(b->stream, b->d_bwt, m, d_counts, &b->stats.kernel_launches);
        DSM_CUDA(cudaMemcpyAsync(out256, d_counts, 256 * 8, cudaMemcpyDeviceToHost, b->stream));
        DSM_CUDA(cudaStreamSynchronize(b->stream));
        dev_free(d_counts, b->stream);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

static int check_pieces_args(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, const char *who)
{
    if (!b->built || b->shard_count <= 1) return b->fail(DSMFM_EINVAL, "%s: needs a built sharded builder", who);
    if (!hist_all || world == 0) return b->fail(DSMFM_EINVAL, "%s: bad histogram table", who);
    // the slices together must hold exactly the symbols of the collection
    for (int c = 0; c < 256; ++c) {
        uint64_t t = 0;
        for (uint32_t r = 0; r < world; ++r) t += hist_all[(size_t)r * 256 + c];
        if (t != b->counts[c]) return b->fail(DSMFM_EINVAL, "%s: slice histograms do not add up to the collection's", who);
    }
    return DSMFM_OK;
}

DSMFM_API uint64_t dsmfm_pieces_bytes(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank)
{
    if (!b || !hist_all || rank > world) return 0;
    try {
        WaveletResult tmp;
        wavelet_prepare(b->index.codetable, tmp);
        const PiecePlan p = plan_pieces(tmp.shape, hist_all, world);
        return rank == world ? p.total_bytes : p.rank_bytes[rank];
    } catch (const CudaError &) {
        return 0;
    }
}

DSMFM_API int dsmfm_build_pieces(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank, void *dst_dev)
{
    API_GUARD(b);
    int rc = check_pieces_args(b, hist_all, world, "dsmfm_build_pieces");
    if (rc) return rc;
    if (rank >= world || !dst_dev || !b->d_bwt) return b->fail(DSMFM_EINVAL, "dsmfm_build_pieces: bad arguments");
    try {
        WaveletResult tmp;
        wavelet_prepare(b->index.codetable, tmp);
        const int m = tmp.shape.n_internal;
        const PiecePlan p = plan_pieces(tmp.shape, hist_all, world);
        uint64_t mine = 0;
        for (int c = 0; c < 256; ++c) mine += hist_all[(size_t)rank * 256 + c];
        if (mine != b->shard_m) return b->fail(DSMFM_EINVAL, "dsmfm_build_pieces: histogram row %u is not this slice's", rank);
        uint8_t *dst = static_cast<uint8_t *>(dst_dev);
        DSM_CUDA(cudaMemsetAsync(dst, 0, p.rank_bytes[rank], b->stream));
        std::vector<uint64_t *> ptrs(m);
        std::vector<uint64_t> base(m);
        for (int v = 0; v < m; ++v) {
            ptrs[v] = reinterpret_cast<uint64_t *>(dst) + p.word_off[(size_t)rank * m + v];
            base[v] = p.bit_off[(size_t)rank * m + v] & 63;
        }
        wavelet_fill_bits(b->stream, b->d_bwt, b->shard_m, tmp.shape, ptrs, base, dst + p.rank_words[rank] * 8,
                          &b->stats.kernel_launches);
        DSM_CUDA(cudaStreamSynchronize(b->stream));
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_assemble_pieces(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, const void *pieces_dev)
{
    API_GUARD(b);
    int rc = check_pieces_args(b, hist_all, world, "dsmfm_assemble_pieces");
    if (rc) return rc;
    if (b->assembled) return b->fail(DSMFM_EINVAL, "dsmfm_assemble_pieces: already assembled");
    if (!pieces_dev) return b->fail(DSMFM_EINVAL, "dsmfm_assemble_pieces: null piece buffer");
    try {
        cudaEvent_t e0, e1;
        DSM_CUDA(cudaEventCreate(&e0));
        DSM_CUDA(cudaEventCreate(&e1));
        DSM_CUDA(cudaEventRecord(e0, b->stream));
        WaveletResult &r = b->wt;
        wavelet_prepare(b->index.codetable, r);
        const int m = r.shape.n_internal;
        if (m > 0) {
            wavelet_alloc(b->stream, r);
            const PiecePlan p = plan_pieces(r.shape, hist_all, world);
            const uint8_t *src = static_cast<const uint8_t *>(pieces_dev);
            std::vector<WtPiece> table;
            std::vector<uint8_t> ch(m, 0), trailers((size_t)world * m);
            for (uint32_t q = 0; q < world; ++q) // first member symbols reported by every rank
                DSM_CUDA(cudaMemcpyAsync(trailers.data() + (size_t)q * m, src + p.rank_byte_off[q] + p.rank_words[q] * 8,
                                         (size_t)m, cudaMemcpyDeviceToHost, b->stream));
            for (int v = 0; v < m; ++v)
                for (uint32_t q = 0; q < world; ++q) {
                    const size_t i = (size_t)q * m + v;
                    if (!p.count[i]) continue;
                    table.push_back(WtPiece{p.rank_byte_off[q] / 8 + p.word_off[i],
                                            reinterpret_cast<uint64_t *>(r.d_sections + r.off_data[v]) + (p.bit_off[i] >> 6),
                                            p.words[i]});
                }
            WtPiece *d_table = static_cast<WtPiece *>(dev_alloc(sizeof(WtPiece) * (table.size() + 1), b->stream));
            DSM_CUDA(cudaMemcpyAsync(d_table, table.data(), sizeof(WtPiece) * table.size(), cudaMemcpyHostToDevice, b->stream));
            launch_wt_merge_pieces(b->stream, reinterpret_cast<const uint64_t *>(src), d_table, (uint32_t)table.size(),
                                   &b->stats.kernel_launches);
            DSM_CUDA(cudaStreamSynchronize(b->stream));
            dev_free(d_table, b->stream);
            for (int v = 0; v < m; ++v) // HuffWT.cpp:8: ch = first symbol of the node's subsequence
                for (uint32_t q = 0; q < world; ++q)
                    if (p.count[(size_t)q * m + v]) {
                        ch[v] = trailers[(size_t)q * m + v];
                        break;
                    }
            DSM_CUDA(cudaMemcpyAsync(r.d_ch, ch.data(), (size_t)m, cudaMemcpyHostToDevice, b->stream));
            wavelet_ranks(b->stream, r, &b->stats.kernel_launches);
        }
        DSM_CUDA(cudaEventRecord(e1, b->stream));
        DSM_CUDA(cudaStreamSynchronize(b->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        b->stats.ms_wt = ms;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    b->assembled = true;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_device_count(void)
{
    int n = 0;
    return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

DSMFM_API void *dsmfm_device_alloc(int device, size_t bytes)
{
    void *p = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

DSMFM_API void dsmfm_device_free(int device, void *p)
{
    if (p && cudaSetDevice(device) == cudaSuccess) cudaFree(p);
}

DSMFM_API int dsmfm_slot_send(dsmfm_builder *b, const dsmfm_text_plan *plan, uint32_t rank, const void *text_src_dev,
                              int dst_device, void *text_dst_dev)
{
    API_GUARD(b);
    if (!plan || rank >= plan->world || !text_src_dev || !text_dst_dev) return b->fail(DSMFM_EINVAL, "dsmfm_slot_send: bad arguments");
    try {
        const size_t bytes = (size_t)plan->slot_words * 8, off = (size_t)rank * bytes;
        const uint8_t *src = static_cast<const uint8_t *>(text_src_dev) + off;
        uint8_t *dst = static_cast<uint8_t *>(text_dst_dev) + off;
        if (dst_device == b->device) {
            if (src != dst) DSM_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, b->stream));
        } else {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, b->device, dst_device) == cudaSuccess && can) {
                const cudaError_t e = cudaDeviceEnablePeerAccess(dst_device, 0); // direct stores over NVLink
                if (e != cudaSuccess) cudaGetLastError();                         // (already enabled)
            }
            DSM_CUDA(cudaMemcpyPeerAsync(dst, dst_device, src, b->device, bytes, b->stream));
        }
        DSM_CUDA(cudaStreamSynchronize(b->stream));
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    }
    return DSMFM_OK;
}

// ---- wavelet tree and BitRank directories built where the BWT slices are --------------------------
// Slice r's members of node v occupy the bits [o, o + c) of the node's vector (o, c from the slices' byte
// histograms).  Builder r OWNS the data words whose first bit lies in that range -- [ceil(o/64), ceil((o+c)/64)) --
// with their Rb entries, and the Rs entries of the superblocks that start in it; the last slice with members also
// owns what lies behind the last bit (BitRank.cpp:97-101: integers = n/64 + 1).  Everything owned follows from the
// slice's own bits plus B = the ones of the slices in front of it (histograms again), except next to a boundary:
// the last owned word may hold bits of later slices, and the Rb entries of a superblock that starts in front of
// the slice need the ones of earlier slices inside that superblock.  Those few words travel as dsmfm_piece_edge.
namespace {
uint64_t ones_of_slice(const WtShape &shape, int v, const uint64_t *hist_row)
{
    uint64_t c = 0;
    for (int s = 0; s < 256; ++s)
        if (shape.info[(size_t)v * 256 + s] == 3u) c += hist_row[s];
    return c;
}

// offsets of every section of the .fmi file (FMIndex::save, FMIndex.cpp:155-217)
void fmi_layout(const WtShape &shape, std::vector<uint64_t> &node_off, std::vector<uint64_t> &data_off,
                std::vector<uint64_t> &rs_off, std::vector<uint64_t> &rb_off, uint64_t &tail_off, uint64_t &total)
{
    uint64_t pos = 1 + 8 + 4 + 2048 + 8 + 256 * 16;
    node_off.assign(shape.nodes.size(), 0);
    data_off.assign(shape.n_internal, 0);
    rs_off.assign(shape.n_internal, 0);
    rb_off.assign(shape.n_internal, 0);
    for (size_t i = 0; i < shape.nodes.size(); ++i) {
        node_off[i] = pos;
        pos += 2;
        const int v = shape.internal_of_node[i];
        if (v < 0) continue;
        const dsmfm_node &nd = shape.nodes[i];
        pos += 8 + 8 + 4 + 4;
        data_off[v] = pos;
        pos += nd.integers * 8;
        rs_off[v] = pos;
        pos += (nd.nbits / 256 + 1) * 8;
        rb_off[v] = pos;
        pos += nd.nbits / 64 + 1;
    }
    tail_off = pos;
    total = pos + 4 + 8 + 1 + 1 + 1 + 4;
}

bool pwrite_all(int fd, const void *p, size_t n, uint64_t off)
{
    const uint8_t *q = static_cast<const uint8_t *>(p);
    while (n) {
        const ssize_t w = ::pwrite(fd, q, n, (off_t)off);
        if (w <= 0) return false;
        q += w;
        n -= (size_t)w;
        off += (uint64_t)w;
    }
    return true;
}

// The owned share (pc) and the edge record (ed) of one vector, from the host copy of the builder's blob.  Returns
// the bytes owned.
uint64_t vec_fetch(const VecPiece &l, uint8_t *h_blob, dsmfm_piece &pc, dsmfm_piece_edge &ed)
{
    pc = dsmfm_piece();
    ed = dsmfm_piece_edge();
    if (!l.c) return 0;
    uint64_t *h_data = reinterpret_cast<uint64_t *>(h_blob + l.off_data);
    pc.word_first = div_up(l.o, 64);
    const uint64_t w_end = l.last ? l.nbits / 64 + 1 : div_up(l.o + l.c, 64);
    pc.word_count = w_end > pc.word_first ? w_end - pc.word_first : 0;
    pc.data = h_data + (pc.word_first - l.G0);
    if (l.dirs) {
        pc.rb_first = pc.word_first;
        pc.rb_count = pc.word_count;
        pc.rs_first = div_up(l.o, 256);
        const uint64_t s_end = l.last ? l.nbits / 256 + 1 : div_up(l.o + l.c, 256);
        pc.rs_count = s_end > pc.rs_first ? s_end - pc.rs_first : 0;
        pc.Rb = h_blob + l.off_rb + (pc.word_first - l.G0);
        pc.Rs = reinterpret_cast<uint64_t *>(h_blob + l.off_rs) + (pc.rs_first - l.G0 / 4);
    }
    ed.count = l.c;
    ed.first_word = l.o / 64;
    ed.last_word = (l.o + l.c - 1) / 64;
    for (int t = 0; t < 4; ++t) {
        const uint64_t fi = ed.first_word - l.G0 + t;
        ed.first[t] = fi < l.words ? h_data[fi] : 0ull;
        const int64_t li = (int64_t)(ed.last_word - l.G0) - 3 + t;
        ed.last[t] = li >= 0 && (uint64_t)li < l.words ? h_data[li] : 0ull;
    }
    return pc.word_count * 8 + pc.rs_count * 8 + pc.rb_count;
}

// Completes the owned words next to the slice boundaries from the edge records of every builder
// (edges[q * stride] is builder q's record of this vector).
void vec_merge(const VecPiece &l, dsmfm_piece &pc, const dsmfm_piece_edge *edges, size_t stride, uint32_t world, uint32_t rank)
{
    if (!l.c) return;
    // what any builder contributes to data word w (first / last windows of its record)
    auto contribution = [&](uint32_t q, uint64_t w) -> uint64_t {
        const dsmfm_piece_edge &e = edges[(size_t)q * stride];
        if (!e.count) return 0ull;
        uint64_t x = 0;
        if (w >= e.first_word && w < e.first_word + 4) x |= e.first[w - e.first_word];
        if (w + 3 >= e.last_word && w <= e.last_word) x |= e.last[w + 3 - e.last_word];
        return x;
    };
    // (a) bits of later slices in the last owned word (and, for tiny slices, in any owned word)
    for (uint32_t q = 0; q < world; ++q) {
        if (q == rank) continue;
        const dsmfm_piece_edge &e = edges[(size_t)q * stride];
        if (!e.count) continue;
        for (int t = 0; t < 4; ++t) {
            const uint64_t wf = e.first_word + t;
            if (wf >= pc.word_first && wf < pc.word_first + pc.word_count) pc.data[wf - pc.word_first] |= e.first[t];
            if (e.last_word + t >= 3) {
                const uint64_t wl = e.last_word - 3 + t;
                if (wl >= pc.word_first && wl < pc.word_first + pc.word_count) pc.data[wl - pc.word_first] |= e.last[t];
            }
        }
    }
    if (!l.dirs) return;
    // (b) Rb of the owned words whose superblock starts in front of the slice
    const uint64_t first_full = 4 * div_up(l.o, 256); // first word of the first superblock that starts inside the slice
    for (uint64_t k = pc.rb_first; k < pc.rb_first + pc.rb_count && k < first_full; ++k) {
        uint32_t sum = 0;
        for (uint64_t w = 4 * (k / 4); w < k; ++w) {
            uint64_t x = 0;
            if (w >= pc.word_first && w < pc.word_first + pc.word_count) {
                x = pc.data[w - pc.word_first];
            } else {
                for (uint32_t q = 0; q < world; ++q) x |= contribution(q, w);
            }
            sum += (uint32_t)__builtin_popcountll(x);
        }
        pc.Rb[k - pc.rb_first] = (uint8_t)sum;
    }
}

// pwrite of the owned share; data_off / rs_off / rb_off: file offsets of the vector's words / Rs / Rb
bool vec_write(int fd, const VecPiece &l, const dsmfm_piece &pc, uint64_t data_off, uint64_t rs_off, uint64_t rb_off)
{
    if (!l.c) return true;
    bool ok = pwrite_all(fd, pc.data, pc.word_count * 8, data_off + pc.word_first * 8);
    if (l.dirs) {
        ok = ok && pwrite_all(fd, pc.Rs, pc.rs_count * 8, rs_off + pc.rs_first * 8);
        ok = ok && pwrite_all(fd, pc.Rb, pc.rb_count, rb_off + pc.rb_first);
    }
    return ok;
}
} // namespace

DSMFM_API int dsmfm_pieces_fetch(dsmfm_builder *b, dsmfm_pieces *out);

DSMFM_API int dsmfm_pieces_build(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank, dsmfm_pieces *out)
{
    API_GUARD(b);
    if (!hist_all || world == 0 || rank >= world) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_build: bad arguments");
    if (!b->built || !b->d_bwt) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_build: nothing built (or already fetched)");
    if (b->ph.built) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_build: already built");
    for (int c = 0; c < 256; ++c) { // the slices together must hold exactly the symbols of the collection
        uint64_t t = 0;
        for (uint32_t r = 0; r < world; ++r) t += hist_all[(size_t)r * 256 + c];
        if (t != b->counts[c]) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_build: slice histograms do not add up to the collection's");
    }
    uint64_t mine = 0;
    for (int c = 0; c < 256; ++c) mine += hist_all[(size_t)rank * 256 + c];
    const uint64_t slice_m = b->shard_count > 1 || b->ext ? b->shard_m : b->index.n;
    if (mine != slice_m) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_build: histogram row %u is not this slice's", rank);
    try {
        cudaStream_t st = b->stream;
        uint32_t *L = &b->stats.kernel_launches;
        cudaEvent_t e0, e1;
        DSM_CUDA(cudaEventCreate(&e0));
        DSM_CUDA(cudaEventCreate(&e1));
        DSM_CUDA(cudaEventRecord(e0, st));
        auto &ph = b->ph;
        WaveletResult tmp;
        wavelet_prepare(b->index.codetable, tmp);
        ph.shape = tmp.shape;
        ph.world = world;
        ph.rank = rank;
        const int m = ph.shape.n_internal;
        const PiecePlan pp = plan_pieces(ph.shape, hist_all, world);
        std::vector<uint64_t> nbits_of(m, 0);
        std::vector<uint32_t> node_of(m, 0);
        for (size_t i = 0; i < ph.shape.nodes.size(); ++i) {
            const int v = ph.shape.internal_of_node[i];
            if (v >= 0) { nbits_of[v] = ph.shape.nodes[i].nbits; node_of[v] = (uint32_t)i; }
        }
        ph.piece.assign(m, dsmfm_piece());
        ph.edge.assign(m, dsmfm_piece_edge());
        ph.vec.assign(m, VecPiece());
        std::vector<uint64_t> ones_before(m, 0);
        size_t blob = 0;
        for (int v = 0; v < m; ++v) {
            const uint64_t c = pp.count[(size_t)rank * m + v];
            bool last = c > 0;
            for (uint32_t q = rank + 1; q < world; ++q)
                if (pp.count[(size_t)q * m + v]) last = false;
            ph.vec[v] = vec_layout(pp.bit_off[(size_t)rank * m + v], c, nbits_of[v], last, true, blob);
            for (uint32_t q = 0; q < rank; ++q) ones_before[v] += ones_of_slice(ph.shape, v, hist_all + (size_t)q * 256);
        }
        const size_t blob_bytes = blob + align8((size_t)(m ? m : 1));
        uint8_t *d_blob = static_cast<uint8_t *>(b->dmalloc(blob_bytes));
        DSM_CUDA(cudaMemsetAsync(d_blob, 0, blob_bytes, st));
        uint8_t *d_ch = d_blob + blob;
        std::vector<uint64_t *> ptrs(m);
        std::vector<uint64_t> base(m);
        uint64_t max_sb = 1;
        for (int v = 0; v < m; ++v) {
            ptrs[v] = reinterpret_cast<uint64_t *>(d_blob + ph.vec[v].off_data);
            base[v] = ph.vec[v].base;
            max_sb = std::max(max_sb, ph.vec[v].nsb);
        }
        wavelet_fill_bits(st, b->d_bwt, slice_m, ph.shape, ptrs, base, d_ch, L);
        uint64_t *d_scratch = static_cast<uint64_t *>(b->dmalloc(sizeof(uint64_t) * (div_up(max_sb, kRankChunk) + 1)));
        for (int v = 0; v < m; ++v)
            if (ph.vec[v].c)
                launch_bitrank(st, ptrs[v], ph.vec[v].nb, reinterpret_cast<uint64_t *>(d_blob + ph.vec[v].off_rs),
                               d_blob + ph.vec[v].off_rb, d_scratch, L, ones_before[v]);
        DSM_CUDA(cudaEventRecord(e1, st));
        DSM_CUDA(cudaStreamSynchronize(st));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        b->stats.ms_wt = ms;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        b->dfree(d_scratch);
        b->dfree(b->d_bwt);
        b->d_bwt = nullptr;
        ph.d_blob = d_blob;
        ph.blob_bytes = blob_bytes;
        ph.ch_off = blob;
        ph.node_of = node_of;
        ph.built = true;
        ph.merged = false;
        if (out) {
            const int rc = dsmfm_pieces_fetch(b, out);
            if (rc) return rc;
        }
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_pieces_fetch(dsmfm_builder *b, dsmfm_pieces *out)
{
    API_GUARD(b);
    if (!out) return DSMFM_EINVAL;
    auto &ph = b->ph;
    if (!ph.built) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_fetch: call dsmfm_pieces_build first");
    try {
        cudaStream_t st = b->stream;
        const int m = ph.shape.n_internal;
        if (!ph.h_blob) {
            cudaEvent_t e0, e1;
            DSM_CUDA(cudaEventCreate(&e0));
            DSM_CUDA(cudaEventCreate(&e1));
            ph.h_blob = static_cast<uint8_t *>(g_pinned.get(ph.blob_bytes));
            ph.h_bytes = ph.blob_bytes;
            DSM_CUDA(cudaEventRecord(e0, st));
            DSM_CUDA(cudaMemcpyAsync(ph.h_blob, ph.d_blob, ph.blob_bytes, cudaMemcpyDeviceToHost, st));
            DSM_CUDA(cudaEventRecord(e1, st));
            DSM_CUDA(cudaStreamSynchronize(st));
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            b->stats.ms_d2h = ms;
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
            b->dfree(ph.d_blob);
            ph.d_blob = nullptr;
        }
        uint64_t held = 0;
        for (int v = 0; v < m; ++v) {
            held += vec_fetch(ph.vec[v], ph.h_blob, ph.piece[v], ph.edge[v]);
            ph.piece[v].node = ph.node_of[v];
            if (ph.vec[v].c) ph.edge[v].ch = ph.h_blob[ph.ch_off + v];
        }
        out->n_internal = (uint32_t)m;
        out->world = ph.world;
        out->rank = ph.rank;
        out->reserved = 0;
        out->bytes = held;
        out->piece = ph.piece.data();
        out->edge = ph.edge.data();
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_pieces_merge(dsmfm_builder *b, const dsmfm_piece_edge *edges_all, uint32_t world)
{
    if (!b || !edges_all) return DSMFM_EINVAL;
    auto &ph = b->ph;
    if (!ph.h_blob || world != ph.world) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_merge: call dsmfm_pieces_build / dsmfm_pieces_fetch first (same world)");
    if (ph.merged) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_merge: already merged");
    const int m = ph.shape.n_internal;
    for (int v = 0; v < m; ++v) vec_merge(ph.vec[v], ph.piece[v], edges_all + v, (size_t)m, world, ph.rank);
    // node symbols (every builder fills the whole table: the one that writes the header needs it)
    for (size_t i = 0; i < ph.shape.nodes.size(); ++i) {
        const int v = ph.shape.internal_of_node[i];
        if (v < 0) continue;
        for (uint32_t q = 0; q < world; ++q) {
            const dsmfm_piece_edge &e = edges_all[(size_t)q * m + v];
            if (e.count) {
                ph.shape.nodes[i].ch = (uint8_t)e.ch;
                break;
            }
        }
    }
    ph.merged = true;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_pieces_index(dsmfm_builder *b, dsmfm_index *out)
{
    if (!b || !out) return DSMFM_EINVAL;
    if (!b->ph.merged) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_index: call dsmfm_pieces_merge first");
    *out = b->index;
    out->n_nodes = (uint32_t)b->ph.shape.nodes.size();
    out->nodes = b->ph.shape.nodes.data();
    out->bwt = nullptr;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_pieces_write(dsmfm_builder *b, const char *path_prefix, int header)
{
    if (!b || !path_prefix) return DSMFM_EINVAL;
    auto &ph = b->ph;
    if (!ph.merged) return b->fail(DSMFM_EINVAL, "dsmfm_pieces_write: call dsmfm_pieces_merge first");
    const std::string name = std::string(path_prefix) + ".fmi"; // TextCollection::FMINDEX_EXTENSION
    const int fd = ::open(name.c_str(), O_WRONLY | O_CREAT, 0644);
    if (fd < 0) return b->fail(DSMFM_EIO, "dsmfm_pieces_write: can not open %s", name.c_str());
    std::vector<uint64_t> node_off, data_off, rs_off, rb_off;
    uint64_t tail_off = 0, total = 0;
    fmi_layout(ph.shape, node_off, data_off, rs_off, rb_off, tail_off, total);
    bool ok = true;
    const int m = ph.shape.n_internal;
    for (int v = 0; v < m && ok; ++v) ok = vec_write(fd, ph.vec[v], ph.piece[v], data_off[v], rs_off[v], rb_off[v]);
    if (header && ok) {
        std::vector<uint8_t> h;
        auto put = [&h](const void *p, size_t n) {
            const uint8_t *q = static_cast<const uint8_t *>(p);
            h.insert(h.end(), q, q + n);
        };
        const uint8_t version = 17; // FMIndex.cpp:51
        const uint64_t bwt_end_pos = 0;
        put(&version, 1);
        put(&b->index.n, 8);
        put(&b->index.samplerate, 4);
        put(b->index.C, sizeof b->index.C);
        put(&bwt_end_pos, 8);
        for (int i = 0; i < 256; ++i) {
            put(&b->index.codetable[i].count, 8);
            put(&b->index.codetable[i].bits, 4);
            put(&b->index.codetable[i].code, 4);
        }
        ok = ok && pwrite_all(fd, h.data(), h.size(), 0);
        const uint32_t b64 = 64, s256 = 256;
        for (size_t i = 0; i < ph.shape.nodes.size() && ok; ++i) {
            const dsmfm_node &nd = ph.shape.nodes[i];
            h.clear();
            put(&nd.leaf, 1);
            put(&nd.ch, 1);
            if (!nd.leaf) {
                put(&nd.nbits, 8);
                put(&nd.integers, 8);
                put(&b64, 4);
                put(&s256, 4);
            }
            ok = ok && pwrite_all(fd, h.data(), h.size(), node_off[i]);
        }
        h.clear();
        const uint8_t z8 = 0;
        const uint32_t z32 = 0;
        put(&b->index.number_of_texts, 4);
        put(&b->index.max_text_length, 8);
        put(&z8, 1);
        put(&z8, 1);
        put(&z8, 1);
        put(&z32, 4);
        ok = ok && pwrite_all(fd, h.data(), h.size(), tail_off);
        ok = ok && ::ftruncate(fd, (off_t)total) == 0;
    }
    ok = (::close(fd) == 0) && ok;
    return ok ? DSMFM_OK : b->fail(DSMFM_EIO, "dsmfm_pieces_write: write error on %s", name.c_str());
}

// ---- .sa samples of a packed-text build (include/dsmfm.h, steps 8-11) ----
// The five vectors of FMIndex::saveSamples (FMIndex.cpp:134-143) and this builder's range of each, in bits:
//   sampled      n bits            [rank_begin, + count)        directories, ones in front: samples of earlier slices
//   suffixes     S * wlen          [S_<r * wlen, + s_r * wlen)  S = samples; S_<r, s_r: of earlier slices / this one
//   suffixDocId  S * wdoc          [S_<r * wdoc, + s_r * wdoc)
//   textLength   D * wlen          documents of this block
//   Doc          D * wdoc          [Z_<r * wdoc, + z_r * wdoc)  Z_<r, z_r: end markers of earlier slices / this one
namespace {
enum { kSaSampled, kSaSuffixes, kSaDocId, kSaTextLength, kSaDoc };

struct SaFileLayout {
    uint64_t data[DSMFM_SA_VECTORS], rs, rb, hdr[DSMFM_SA_VECTORS], total;
};

// offsets in the .sa file (dsmfm_builder::make_sa_image): BitRank header and arrays, then four BlockArrays of
// 16 header bytes and count * width / 64 + 1 words each
SaFileLayout sa_file_layout(uint64_t n, uint64_t S, uint64_t D, unsigned wlen, unsigned wdoc)
{
    SaFileLayout f;
    f.hdr[kSaSampled] = 0;
    f.data[kSaSampled] = 24;
    f.rs = f.data[kSaSampled] + (n / 64 + 1) * 8;
    f.rb = f.rs + (n / 256 + 1) * 8;
    uint64_t p = f.rb + n / 64 + 1;
    const uint64_t count[DSMFM_SA_VECTORS] = {0, S, S, D, D};
    const unsigned width[DSMFM_SA_VECTORS] = {0, wlen, wdoc, wlen, wdoc};
    for (int i = 1; i < DSMFM_SA_VECTORS; ++i) {
        f.hdr[i] = p;
        f.data[i] = p + 16;
        p += 16 + (count[i] * width[i] / 64 + 1) * 8;
    }
    f.total = p;
    return f;
}
} // namespace

DSMFM_API int dsmfm_sa_slice_info(dsmfm_builder *b, dsmfm_sa_info *out)
{
    if (!b || !out) return DSMFM_EINVAL;
    if (!b->sah.ready)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_slice_info: needs dsmfm_build_packed on a builder with DSMFM_FLAG_KEEP_SA");
    *out = b->sah.info;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_sa_pieces_build(dsmfm_builder *b, const dsmfm_sa_info *infos_all, uint32_t world, uint32_t rank,
                                    dsmfm_piece_edge *edges_out)
{
    API_GUARD(b);
    auto &sa = b->sah;
    if (!sa.ready)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: needs dsmfm_build_packed on a builder with DSMFM_FLAG_KEEP_SA");
    if (sa.built) return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: already built");
    if (!infos_all || !edges_out) return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: bad arguments");
    if (world != sa.world || rank >= world)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: world %u / rank %u, the build has %u blocks", world, rank, sa.world);
    const dsmfm_sa_info &me = infos_all[rank];
    if (me.samples != sa.info.samples || me.ends != sa.info.ends || me.documents != sa.info.documents)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: record %u is not this builder's", rank);
    const uint64_t n = b->index.n, D = b->index.number_of_texts;
    uint64_t S = 0, S_before = 0, Z_before = 0, D_before = 0, docs = 0, ends = 0;
    for (uint32_t q = 0; q < world; ++q) {
        if (q < rank) {
            S_before += infos_all[q].samples;
            Z_before += infos_all[q].ends;
            D_before += infos_all[q].documents;
        }
        S += infos_all[q].samples;
        docs += infos_all[q].documents;
        ends += infos_all[q].ends;
    }
    if (docs != D || ends != D)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_build: the records hold %llu documents and %llu end markers, the collection %llu",
                       (unsigned long long)docs, (unsigned long long)ends, (unsigned long long)D);
    try {
        cudaStream_t st = b->stream;
        uint32_t *L = &b->stats.kernel_launches;
        const unsigned wlen = ceil_log2(b->index.max_text_length), wdoc = ceil_log2(D);
        const uint64_t s_r = sa.info.samples, z_r = sa.info.ends, d_r = sa.info.documents, m = b->shard_m;
        // each vector: (bit offset, bit count, total bits) of this builder; the last builder with bits owns the tail
        const uint64_t o[DSMFM_SA_VECTORS] = {b->shard_rank_begin, S_before * wlen, S_before * wdoc, D_before * wlen, Z_before * wdoc};
        const uint64_t c[DSMFM_SA_VECTORS] = {m, s_r * wlen, s_r * wdoc, d_r * wlen, z_r * wdoc};
        const uint64_t total[DSMFM_SA_VECTORS] = {n, S * wlen, S * wdoc, D * wlen, D * wdoc};
        size_t blob = 0;
        for (int i = 0; i < DSMFM_SA_VECTORS; ++i) {
            const bool last = c[i] > 0 && o[i] + c[i] == total[i];
            sa.vec[i] = vec_layout(o[i], c[i], total[i], last, i == kSaSampled, blob);
        }
        uint8_t *d_blob = static_cast<uint8_t *>(b->dmalloc(blob));
        DSM_CUDA(cudaMemsetAsync(d_blob, 0, blob, st));
        auto data = [&](int i) { return reinterpret_cast<uint64_t *>(d_blob + sa.vec[i].off_data); };
        const VecPiece &vs = sa.vec[kSaSampled];
        DSM_CUDA(cudaMemcpyAsync(data(kSaSampled), sa.d_sampled, vs.words * 8, cudaMemcpyDeviceToDevice, st));
        // directories of `sampled` (final: the samples of earlier slices in front) and, local, of the end markers
        const uint64_t ends_sb = m / 256 + 1;
        uint64_t *d_ends_rs = static_cast<uint64_t *>(b->dmalloc(ends_sb * 8));
        uint8_t *d_ends_rb = static_cast<uint8_t *>(b->dmalloc(m / 64 + 1 + 8));
        uint64_t *d_scratch =
            static_cast<uint64_t *>(b->dmalloc(sizeof(uint64_t) * (div_up(std::max(vs.nsb, ends_sb), kRankChunk) + 1)));
        const uint64_t *sampled_rs = reinterpret_cast<const uint64_t *>(d_blob + vs.off_rs);
        const uint8_t *sampled_rb = d_blob + vs.off_rb;
        if (m) {
            launch_bitrank(st, data(kSaSampled), vs.nb, reinterpret_cast<uint64_t *>(d_blob + vs.off_rs), d_blob + vs.off_rb,
                           d_scratch, L, S_before);
            launch_bitrank(st, sa.d_ends, m, d_ends_rs, d_ends_rb, d_scratch, L, 0);
        }
        // the fields: offset and document of every sample, document of every end marker, length of every document
        launch_sa_emit64(st, b->d_sa, b->d_sa_hi, b->pos_lo_bits, data(kSaSampled), sampled_rs, sampled_rb, vs.base, S_before,
                         m, sa.d_doc_end, (uint32_t)D, sa.slot_syms, data(kSaDocId), sa.vec[kSaDocId].base, wdoc,
                         data(kSaSuffixes), sa.vec[kSaSuffixes].base, wlen, L);
        launch_sa_emit64(st, b->d_sa, b->d_sa_hi, b->pos_lo_bits, sa.d_ends, d_ends_rs, d_ends_rb, 0, 0, m, sa.d_doc_end,
                         (uint32_t)D, sa.slot_syms, data(kSaDoc), sa.vec[kSaDoc].base, wdoc, nullptr, 0, 0, L);
        launch_sa_lengths(st, sa.d_doc_end, D_before, d_r, sa.slot_syms, data(kSaTextLength), sa.vec[kSaTextLength].base,
                          wlen, L);
        sa.h_blob.resize(blob);
        DSM_CUDA(cudaMemcpyAsync(sa.h_blob.data(), d_blob, blob, cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaStreamSynchronize(st));
        for (void *p : {(void *)d_blob, (void *)d_ends_rs, (void *)d_ends_rb, (void *)d_scratch, (void *)sa.d_sampled,
                        (void *)sa.d_ends, (void *)sa.d_doc_end, (void *)b->d_sa, (void *)b->d_sa_hi})
            b->dfree(p);
        sa.d_sampled = sa.d_ends = sa.d_doc_end = nullptr;
        b->d_sa = nullptr;
        b->d_sa_hi = nullptr;
        for (int i = 0; i < DSMFM_SA_VECTORS; ++i) {
            vec_fetch(sa.vec[i], sa.h_blob.data(), sa.piece[i], sa.edge[i]);
            edges_out[i] = sa.edge[i];
        }
        sa.rank = rank;
        sa.samples = S;
        sa.wlen = wlen;
        sa.wdoc = wdoc;
        sa.built = true;
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_sa_pieces_merge(dsmfm_builder *b, const dsmfm_piece_edge *edges_all, uint32_t world)
{
    if (!b || !edges_all) return DSMFM_EINVAL;
    auto &sa = b->sah;
    if (!sa.built || world != sa.world)
        return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_merge: call dsmfm_sa_pieces_build first (same world)");
    if (sa.merged) return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_merge: already merged");
    for (int i = 0; i < DSMFM_SA_VECTORS; ++i) vec_merge(sa.vec[i], sa.piece[i], edges_all + i, DSMFM_SA_VECTORS, world, sa.rank);
    sa.merged = true;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_sa_pieces_write(dsmfm_builder *b, const char *path_prefix, int header)
{
    if (!b || !path_prefix) return DSMFM_EINVAL;
    auto &sa = b->sah;
    if (!sa.merged) return b->fail(DSMFM_EINVAL, "dsmfm_sa_pieces_write: call dsmfm_sa_pieces_merge first");
    const std::string name = std::string(path_prefix) + ".sa"; // FMIndex.cpp:131
    const int fd = ::open(name.c_str(), O_WRONLY | O_CREAT, 0644);
    if (fd < 0) return b->fail(DSMFM_EIO, "dsmfm_sa_pieces_write: can not open %s", name.c_str());
    const uint64_t n = b->index.n, D = b->index.number_of_texts;
    const SaFileLayout f = sa_file_layout(n, sa.samples, D, sa.wlen, sa.wdoc);
    bool ok = true;
    for (int i = 0; i < DSMFM_SA_VECTORS && ok; ++i)
        ok = vec_write(fd, sa.vec[i], sa.piece[i], f.data[i], f.rs, f.rb);
    if (header && ok) {
        const uint64_t integers = n / 64 + 1; // BitRank::integers = ceil((n+1)/64)
        const uint32_t b64 = 64, s256 = 256;
        uint8_t h[24];
        std::memcpy(h, &n, 8);
        std::memcpy(h + 8, &integers, 8);
        std::memcpy(h + 16, &b64, 4);
        std::memcpy(h + 20, &s256, 4);
        ok = pwrite_all(fd, h, sizeof h, 0);
        const uint64_t count[DSMFM_SA_VECTORS] = {0, sa.samples, sa.samples, D, D};
        const uint64_t width[DSMFM_SA_VECTORS] = {0, sa.wlen, sa.wdoc, sa.wlen, sa.wdoc};
        const uint64_t zero = 0;
        for (int i = 1; i < DSMFM_SA_VECTORS && ok; ++i) {
            const uint64_t bh[2] = {count[i], width[i]}; // BlockArray::Save (BlockArray.h:54-64)
            ok = pwrite_all(fd, bh, sizeof bh, f.hdr[i]);
            // a vector without bits is its one zero word, which no builder owns
            if (ok && count[i] * width[i] == 0) ok = pwrite_all(fd, &zero, 8, f.data[i]);
        }
        ok = ok && ::ftruncate(fd, (off_t)f.total) == 0;
    }
    ok = (::close(fd) == 0) && ok;
    return ok ? DSMFM_OK : b->fail(DSMFM_EIO, "dsmfm_sa_pieces_write: write error on %s", name.c_str());
}

DSMFM_API int dsmfm_fetch(dsmfm_builder *b, dsmfm_index *out)
{
    API_GUARD(b);
    if (!b->built) return b->fail(DSMFM_EINVAL, "dsmfm_fetch: nothing built");
    if (b->shard_count > 1 && !b->assembled)
        return b->fail(DSMFM_EINVAL, "dsmfm_fetch: a sharded builder holds a slice only; call dsmfm_assemble on one of them");
    try {
        const double t0 = now_ms();
        if (!b->fetched) b->fetch();
        b->stats.ms_wall_fetch = (float)(now_ms() - t0);
    } catch (const CudaError &e) {
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    if (out) *out = b->index;
    return DSMFM_OK;
}

DSMFM_API int dsmfm_finish(dsmfm_builder *b, dsmfm_index *out)
{
    int rc = dsmfm_build_device(b);
    if (rc) return rc;
    return dsmfm_fetch(b, out);
}

DSMFM_API int dsmfm_copy_sa(dsmfm_builder *b, uint32_t *out, uint64_t first, uint64_t count)
{
    API_GUARD(b);
    if (!b->d_sa) return b->fail(DSMFM_EINVAL, "dsmfm_copy_sa: needs DSMFM_FLAG_KEEP_SA and a finished build");
    if (b->shard_count > 1) return b->fail(DSMFM_EINVAL, "dsmfm_copy_sa: sharded builders export their slice with dsmfm_shard_export");
    if (!out || first > b->index.n || count > b->index.n - first) return b->fail(DSMFM_EINVAL, "dsmfm_copy_sa: range out of bounds");
    cudaError_t e = cudaMemcpy(out, b->d_sa + first, count * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return b->fail(DSMFM_ECUDA, "dsmfm_copy_sa: %s", cudaGetErrorString(e));
    return DSMFM_OK;
}

static int ensure_sa_image(dsmfm_builder *b, const char *who)
{
    if (!b->built || !b->d_sa || !b->d_doc_end || !b->d_bwt)
        return b->fail(DSMFM_EINVAL, "%s: needs a finished, unsharded build with DSMFM_FLAG_KEEP_SA", who);
    if (!b->sa_image.empty()) return DSMFM_OK;
    try {
        b->make_sa_image();
    } catch (const CudaError &e) {
        b->sa_image.clear();
        return b->fail_cuda(e);
    } catch (const std::bad_alloc &) {
        b->sa_image.clear();
        return b->fail(DSMFM_ENOMEM, "host allocation failed");
    }
    return DSMFM_OK;
}

DSMFM_API uint64_t dsmfm_sa_size(dsmfm_builder *b)
{
    if (!b) return 0;
    cudaSetDevice(b->device);
    return ensure_sa_image(b, "dsmfm_sa_size") == DSMFM_OK ? b->sa_image.size() : 0;
}

DSMFM_API int dsmfm_sa_serialize(dsmfm_builder *b, uint8_t *out, uint64_t out_cap)
{
    API_GUARD(b);
    int rc = ensure_sa_image(b, "dsmfm_sa_serialize");
    if (rc) return rc;
    if (!out || out_cap < b->sa_image.size()) return b->fail(DSMFM_EINVAL, "dsmfm_sa_serialize: buffer too small");
    std::memcpy(out, b->sa_image.data(), b->sa_image.size());
    return DSMFM_OK;
}

DSMFM_API int dsmfm_write_sa(dsmfm_builder *b, const char *path_prefix)
{
    API_GUARD(b);
    if (!path_prefix) return DSMFM_EINVAL;
    int rc = ensure_sa_image(b, "dsmfm_write_sa");
    if (rc) return rc;
    const std::string name = std::string(path_prefix) + ".sa"; // FMIndex.cpp:131
    FILE *f = std::fopen(name.c_str(), "wb");
    if (!f) return b->fail(DSMFM_EIO, "dsmfm_write_sa: can not open %s", name.c_str());
    const bool ok = std::fwrite(b->sa_image.data(), 1, b->sa_image.size(), f) == b->sa_image.size() && std::fflush(f) == 0;
    std::fclose(f);
    return ok ? DSMFM_OK : b->fail(DSMFM_EIO, "dsmfm_write_sa: write error");
}

DSMFM_API int dsmfm_get_stats(const dsmfm_builder *b, dsmfm_stats *out)
{
    if (!b || !out) return DSMFM_EINVAL;
    *out = b->stats;
    return DSMFM_OK;
}

DSMFM_API const char *dsmfm_last_error(const dsmfm_builder *b)
{
    return b ? b->err.c_str() : g_create_error.c_str();
}

DSMFM_API uint64_t dsmfm_dbg_guard_violations(void) { return g_guard_violations.load(); }

DSMFM_API int dsmfm_release_cached(int device)
{
    g_pinned.trim();
    g_fasta_arena.trim(device);
    g_blocks.trim(device);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess) return DSMFM_ECUDA;
    for (int d = 0; d < ndev; ++d) {
        if (device >= 0 && d != device) continue;
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, d) == cudaSuccess) {
            cudaSetDevice(d);
            cudaDeviceSynchronize();
            cudaMemPoolTrimTo(pool, 0);
        }
    }
    return DSMFM_OK;
}

DSMFM_API void dsmfm_destroy(dsmfm_builder *b)
{
    if (!b) return;
    trace("destroy: begin");
    cudaSetDevice(b->device);
    cudaStreamSynchronize(b->stream);
    b->release_device();
    g_pinned.put(b->h_bwt);
    for (int i = 0; i < 2; ++i) {
        g_pinned.put(b->stage[i]);
        if (b->stage_free[i]) cudaEventDestroy(b->stage_free[i]);
    }
    if (b->own_stream) cudaStreamDestroy(b->stream);
    delete b;
    trace("destroy: done");
}

// ---- serialisation: FMIndex::save, FMIndex.cpp:155-217 ---------------------------------------

namespace {
struct Sink {
    FILE *f = nullptr;
    uint8_t *mem = nullptr;
    uint64_t cap = 0, pos = 0;
    bool ok = true;
    void put(const void *p, size_t n)
    {
        if (!ok) return;
        if (f) {
            if (n && std::fwrite(p, 1, n, f) != n) ok = false;
        } else if (mem) {
            if (pos + n > cap) { ok = false; return; }
            std::memcpy(mem + pos, p, n);
        }
        pos += n;
    }
};

void serialize(const dsmfm_index *idx, Sink &s)
{
    const uint8_t version = 17; // FMIndex.cpp:51
    const uint64_t bwt_end_pos = 0; // never computed on the builder path (FMIndex.cpp:95)
    s.put(&version, 1);
    s.put(&idx->n, 8);
    s.put(&idx->samplerate, 4);
    s.put(idx->C, sizeof idx->C);
    s.put(&bwt_end_pos, 8);
    for (int i = 0; i < 256; ++i) { // TCodeEntry::save, HuffWT.h:37-45
        s.put(&idx->codetable[i].count, 8);
        s.put(&idx->codetable[i].bits, 4);
        s.put(&idx->codetable[i].code, 4);
    }
    const uint32_t b64 = 64, s256 = 256;
    for (uint32_t i = 0; i < idx->n_nodes; ++i) { // HuffWT::save pre-order, HuffWT.cpp:73-86
        const dsmfm_node &nd = idx->nodes[i];
        s.put(&nd.leaf, 1);
        s.put(&nd.ch, 1);
        if (nd.leaf) continue;
        s.put(&nd.nbits, 8); // BitRank::save, BitRank.cpp:134-151
        s.put(&nd.integers, 8);
        s.put(&b64, 4);
        s.put(&s256, 4);
        s.put(nd.data, nd.integers * 8);
        s.put(nd.Rs, (nd.nbits / 256 + 1) * 8);
        s.put(nd.Rb, nd.nbits / 64 + 1);
    }
    const uint8_t z8 = 0;
    const uint32_t z32 = 0;
    s.put(&idx->number_of_texts, 4);
    s.put(&idx->max_text_length, 8);
    s.put(&z8, 1);  // no names   (FMIndex.cpp:190-196)
    s.put(&z8, 1);  // no text    (FMIndex.cpp:198-204)
    s.put(&z8, 1);  // colorCoded (FMIndex.cpp:207)
    s.put(&z32, 4); // rotationLength
}
} // namespace

DSMFM_API uint64_t dsmfm_fmi_size(const dsmfm_index *idx)
{
    if (!idx) return 0;
    Sink s;
    serialize(idx, s);
    return s.pos;
}

DSMFM_API int dsmfm_fmi_serialize(const dsmfm_index *idx, uint8_t *out, uint64_t out_cap)
{
    if (!idx || !out) return DSMFM_EINVAL;
    Sink s;
    s.mem = out;
    s.cap = out_cap;
    serialize(idx, s);
    return s.ok ? DSMFM_OK : DSMFM_EINVAL;
}

DSMFM_API int dsmfm_write_fmi(const dsmfm_index *idx, const char *path_prefix)
{
    if (!idx || !path_prefix) return DSMFM_EINVAL;
    const std::string name = std::string(path_prefix) + ".fmi"; // TextCollection::FMINDEX_EXTENSION
    Sink s;
    trace("write_fmi: begin");
    s.f = std::fopen(name.c_str(), "wb");
    if (!s.f) return DSMFM_EIO;
    serialize(idx, s);
    if (std::fflush(s.f) != 0) s.ok = false;
    std::fclose(s.f);
    trace("write_fmi: file written");
    return s.ok ? DSMFM_OK : DSMFM_EIO;
}

// ---- kernel-level test entry points ------------------------------------------------------

DSMFM_API int dsmfm_dbg_radix_sort(int device, uint64_t *keys, uint32_t *vals, uint64_t n, int begin_bit, int end_bit)
{
    if (!keys || !vals || begin_bit < 0 || end_bit > 64 || begin_bit > end_bit) return DSMFM_EINVAL;
    if (cudaSetDevice(device < 0 ? 0 : device) != cudaSuccess) return DSMFM_ECUDA;
    if (n == 0) return DSMFM_OK;
    uint64_t *ka = nullptr, *kb = nullptr;
    uint32_t *va = nullptr, *vb = nullptr;
    RadixWorkspace ws;
    int rc = DSMFM_OK;
    try {
        DSM_CUDA(cudaMalloc(&ka, n * 8));
        DSM_CUDA(cudaMalloc(&kb, n * 8));
        DSM_CUDA(cudaMalloc(&va, n * 4));
        DSM_CUDA(cudaMalloc(&vb, n * 4));
        ws.allocate(n);
        DSM_CUDA(cudaMemcpy(ka, keys, n * 8, cudaMemcpyHostToDevice));
        DSM_CUDA(cudaMemcpy(va, vals, n * 4, cudaMemcpyHostToDevice));
        const int p = radix_sort_pairs(nullptr, ws, ka, va, kb, vb, n, begin_bit, end_bit, false, nullptr);
        DSM_CUDA(cudaDeviceSynchronize());
        DSM_CUDA(cudaMemcpy(keys, (p & 1) ? kb : ka, n * 8, cudaMemcpyDeviceToHost));
        DSM_CUDA(cudaMemcpy(vals, (p & 1) ? vb : va, n * 4, cudaMemcpyDeviceToHost));
    } catch (const CudaError &e) {
        g_create_error = std::string("dsmfm_dbg_radix_sort: ") + cudaGetErrorString(e.code) + " in " + e.what;
        rc = DSMFM_ECUDA;
    }
    ws.release();
    cudaFree(ka); cudaFree(kb); cudaFree(va); cudaFree(vb);
    return rc;
}

DSMFM_API int dsmfm_dbg_initial_sort(int device, const uint8_t *docs, uint64_t n, int first_key_bits,
                                     const uint64_t *word_cuts, uint32_t ncuts, uint64_t *keys, uint64_t *hist,
                                     uint64_t *sorted_keys, uint32_t *sa, uint32_t *head, uint32_t *diff, uint8_t *bwt,
                                     uint64_t *remaining, int *bits_out, int *first_syms_out, int *carry_out)
{
    // everything the caller hands in is checked before anything is launched
    if (!docs || !keys || !hist || !sorted_keys || !sa || !head || !diff || !bwt || !remaining || !bits_out ||
        !first_syms_out || !carry_out || (ncuts && !word_cuts))
        return DSMFM_EINVAL;
    if (n == 0 || n >= (1ull << 32) - kRefCap - 64 || docs[n - 1] != 0 || docs[0] == 0) return DSMFM_EINVAL;
    uint64_t counts[256] = {};
    for (uint64_t i = 0; i < n; ++i) {
        ++counts[docs[i]];
        if (i && docs[i] == 0 && docs[i - 1] == 0) return DSMFM_EINVAL; // an empty document
    }
    uint8_t code_map[256], inv_map[256] = {};
    const int bits = alphabet_of(counts, code_map, nullptr);
    for (int c = 1; c < 256; ++c)
        if (code_map[c]) inv_map[code_map[c]] = (uint8_t)c;
    const int spw = 64 / bits;
    const uint64_t text_words = div_up(n, spw), nwords = text_words + 8;
    for (uint32_t k = 0; k < ncuts; ++k)
        if (word_cuts[k] == 0 || word_cuts[k] >= text_words || (k && word_cuts[k] <= word_cuts[k - 1])) return DSMFM_EINVAL;
    int first_syms = 0;
    bool carry = false;
    first_key_shape(bits, n, first_key_bits, &first_syms, &carry);
    const int key_bits = first_syms * bits;
    if (cudaSetDevice(device < 0 ? 0 : device) != cudaSuccess) return DSMFM_ECUDA;

    const uint64_t hw = head_words_for(n), out_words = div_up(n, 32);
    uint8_t *d_raw = nullptr, *d_map = nullptr, *d_inv = nullptr, *d_bwt = nullptr;
    uint64_t *d_packed = nullptr, *ka = nullptr, *kb = nullptr;
    uint32_t *va = nullptr, *vb = nullptr, *d_head = nullptr, *d_diff = nullptr;
    unsigned long long *d_rem = nullptr;
    RadixWorkspace ws;
    int rc = DSMFM_OK;
    try {
        DSM_CUDA(cudaMalloc(&d_raw, n + 64));
        DSM_CUDA(cudaMalloc(&d_map, 256));
        DSM_CUDA(cudaMalloc(&d_inv, 256));
        DSM_CUDA(cudaMalloc(&d_packed, nwords * 8));
        DSM_CUDA(cudaMalloc(&ka, n * 8));
        DSM_CUDA(cudaMalloc(&kb, n * 8));
        DSM_CUDA(cudaMalloc(&va, n * 4 + 16));
        DSM_CUDA(cudaMalloc(&vb, n * 4 + 16));
        DSM_CUDA(cudaMalloc(&d_head, hw * 4));
        DSM_CUDA(cudaMalloc(&d_diff, hw * 4));
        DSM_CUDA(cudaMalloc(&d_bwt, n + 64));
        DSM_CUDA(cudaMalloc(&d_rem, 128 * 8));
        ws.allocate(n);
        DSM_CUDA(cudaMemcpy(d_raw, docs, n, cudaMemcpyHostToDevice));
        DSM_CUDA(cudaMemcpy(d_map, code_map, 256, cudaMemcpyHostToDevice));
        DSM_CUDA(cudaMemcpy(d_inv, inv_map, 256, cudaMemcpyHostToDevice));
        // a word read before it is packed shows up as a wrong key, not as a lucky zero
        DSM_CUDA(cudaMemset(d_packed, 0xa5, nwords * 8));
        DSM_CUDA(cudaMemset(ws.hist, 0, sizeof(uint64_t) * kMaxPasses * kRadix));
        if (ncuts == 0) { // build(): the whole text in one go
            launch_pack(nullptr, bits, d_raw, n, d_map, d_packed, nwords, nullptr);
            launch_make_keys_hist(nullptr, bits, d_packed, n, ka, first_syms, carry, ws.hist, nullptr);
        } else { // append_pipelined(): word range by word range
            uint64_t keyed_to = 0;
            for (uint32_t k = 0; k <= ncuts; ++k) {
                const uint64_t w0 = k ? word_cuts[k - 1] : 0;
                const bool last = k == ncuts;
                const uint64_t wn = (last ? nwords : word_cuts[k]) - w0;
                const uint64_t len = last ? n - w0 * spw : wn * spw;
                keyed_to = pack_and_key_range(nullptr, bits, d_raw + w0 * spw, len, d_map, d_packed, w0, wn, last, n,
                                              ka, first_syms, carry, ws.hist, keyed_to, nullptr);
            }
        }
        DSM_CUDA(cudaMemcpy(keys, ka, n * 8, cudaMemcpyDeviceToHost));
        DSM_CUDA(cudaMemcpy(hist, ws.hist, sizeof(uint64_t) * kMaxPasses * kRadix, cudaMemcpyDeviceToHost));
        const int p = radix_sort_pairs(nullptr, ws, ka, va, kb, vb, n, 0, key_bits, true, nullptr, nullptr, nullptr, true);
        uint64_t *sk = (p & 1) ? kb : ka;
        uint32_t *sv = (p & 1) ? vb : va;
        DSM_CUDA(cudaMemset(d_rem, 0, 128 * 8));
        launch_heads(nullptr, bits, sk, n, d_head, hw, d_rem, key_bits, d_inv, carry ? d_bwt : nullptr, nullptr, 0,
                     carry ? d_diff : nullptr, nullptr);
        DSM_CUDA(cudaDeviceSynchronize());
        unsigned long long h_rem[64];
        DSM_CUDA(cudaMemcpy(h_rem, d_rem, sizeof h_rem, cudaMemcpyDeviceToHost));
        DSM_CUDA(cudaMemcpy(sorted_keys, sk, n * 8, cudaMemcpyDeviceToHost));
        DSM_CUDA(cudaMemcpy(sa, sv, n * 4, cudaMemcpyDeviceToHost));
        DSM_CUDA(cudaMemcpy(head, d_head, out_words * 4, cudaMemcpyDeviceToHost));
        if (carry) {
            DSM_CUDA(cudaMemcpy(diff, d_diff, out_words * 4, cudaMemcpyDeviceToHost));
            DSM_CUDA(cudaMemcpy(bwt, d_bwt, n, cudaMemcpyDeviceToHost));
        }
        *remaining = 0;
        for (int i = 0; i < 64; ++i) *remaining += h_rem[i];
        *bits_out = bits;
        *first_syms_out = first_syms;
        *carry_out = carry ? 1 : 0;
    } catch (const CudaError &e) {
        g_create_error = std::string("dsmfm_dbg_initial_sort: ") + cudaGetErrorString(e.code) + " in " + e.what;
        rc = DSMFM_ECUDA;
    }
    ws.release();
    cudaFree(d_raw); cudaFree(d_map); cudaFree(d_inv); cudaFree(d_packed); cudaFree(ka); cudaFree(kb);
    cudaFree(va); cudaFree(vb); cudaFree(d_head); cudaFree(d_diff); cudaFree(d_bwt); cudaFree(d_rem);
    return rc;
}

namespace {
struct DbgIndex {
    WaveletResult wt;
    dsmfm_index index;
};
}

DSMFM_API int dsmfm_dbg_wavelet(int device, const uint8_t *seq, uint64_t n, dsmfm_index *out, void **owner)
{
    if (!seq || !out || !owner || n == 0) return DSMFM_EINVAL;
    if (cudaSetDevice(device < 0 ? 0 : device) != cudaSuccess) return DSMFM_ECUDA;
    DbgIndex *d = new DbgIndex();
    std::memset(&d->index, 0, sizeof d->index);
    uint8_t *d_seq = nullptr;
    uint64_t *d_counts = nullptr;
    int rc = DSMFM_OK;
    try {
        DSM_CUDA(cudaMalloc(&d_seq, n + 64));
        DSM_CUDA(cudaMalloc(&d_counts, 256 * 8));
        DSM_CUDA(cudaMemcpy(d_seq, seq, n, cudaMemcpyHostToDevice));
        DSM_CUDA(cudaMemset(d_counts, 0, 256 * 8));
        launch_byte_hist(nullptr, d_seq, n, d_counts, nullptr);
        uint64_t counts[256];
        DSM_CUDA(cudaMemcpy(counts, d_counts, sizeof counts, cudaMemcpyDeviceToHost));
        d->index.n = n;
        d->index.samplerate = DSMFM_DEFAULT_SAMPLERATE;
        d->index.C[0] = 0;
        for (int i = 1; i < 256; ++i) d->index.C[i] = d->index.C[i - 1] + counts[i - 1];
        if (build_codetable(counts, d->index.codetable) > 32)
            throw CudaError{cudaErrorInvalidValue, "Huffman code longer than 32 bits (the .fmi code field holds 32)", __FILE__, __LINE__};
        wavelet_build_device(nullptr, d_seq, n, d->index.codetable, d->wt, nullptr, nullptr);
        wavelet_fetch(nullptr, d->wt);
        d->index.n_nodes = (uint32_t)d->wt.shape.nodes.size();
        d->index.nodes = d->wt.shape.nodes.data();
    } catch (const CudaError &e) {
        g_create_error = std::string("dsmfm_dbg_wavelet: ") + cudaGetErrorString(e.code) + " in " + e.what;
        rc = DSMFM_ECUDA;
    }
    cudaFree(d_seq);
    cudaFree(d_counts);
    if (rc) {
        d->wt.release();
        delete d;
        return rc;
    }
    *out = d->index;
    *owner = d;
    return DSMFM_OK;
}

DSMFM_API void dsmfm_dbg_free_index(void *owner)
{
    DbgIndex *d = static_cast<DbgIndex *>(owner);
    if (!d) return;
    d->wt.release();
    delete d;
}

} // extern "C"
