// search.cu -- the query half of the index on the GPU (sm_100a): what the mining client asks of an .fmi.
//
// Replaces, for batches of queries, FMIndex::LF / getL (FMIndex.h:84-102) over HuffWT::rank / access
// (HuffWT.h:66-83, 125-157) and BitRank::rank (BitRank.cpp:191-195) -- the only index operations
// EnumerateQuery performs while it walks the suffix trie (Query.h:37-45, EnumerateQuery.cpp:39-58, 105-149).
// The wavelet tree is used in the layout the builder writes and the reference loads (per internal node: bit
// words, Rs per 256 bits, Rb per 64 bits), resident in HBM; one thread answers one query by walking the
// Huffman code of its symbol from the root, three small reads per level.  Indices wrap like the reference's
// unsigned longs: a rank "up to position -1" is 0 because BitRank::rank pre-increments its argument.
#include "common.cuh"
#include "../../include/dsmfm.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <unistd.h>
#include <cstring>
#include <new>
#include <string>
#include <vector>

namespace dsmfm {

namespace {

struct QNode {
    const uint64_t *data; // BitRank::data
    const uint64_t *Rs;   // ones in front of every 256-bit superblock
    const uint8_t *Rb;    // ones in front of every word inside its superblock
    uint64_t nbits;       // length of the node's bit vector: every position handed to it is clamped to this
    int32_t left, right;  // children in the node table
    uint8_t leaf, ch;
    uint8_t pad[6];
};

struct QIndex {
    uint64_t n;
    uint64_t C[257];     // C[256] = n: the reference reads C[c+1] (FMIndex.h:86)
    uint32_t code[256];  // Huffman code of a symbol, first branch in bit 0
    uint8_t present[256];
    QNode nodes[512];
};

// ones among the first `cnt` bits = BitRank::rank(cnt - 1)
__device__ __forceinline__ uint64_t ones_before(const QNode &nd, uint64_t cnt)
{
    return __ldg(nd.Rs + (cnt >> 8)) + __ldg(nd.Rb + (cnt >> 6)) +
           (uint64_t)__popcll(__ldg(nd.data + (cnt >> 6)) & ((1ull << (cnt & 63)) - 1));
}

// HuffWT::rank(c, i): occurrences of c in [0, i]
__device__ __forceinline__ uint64_t wt_rank(const QIndex *__restrict__ x, uint32_t c, uint64_t i)
{
    if (!x->present[c]) return 0;
    uint64_t cnt = i + 1; // positions considered; 0 for i = (ulong)-1
    cnt = cnt < x->n ? cnt : x->n; // i >= n counts as n - 1 also when the root is a leaf (one symbol), not only below it
    uint32_t code = x->code[c];
    const QNode *t = &x->nodes[0];
    while (!t->leaf) {
        // positions behind the node's last bit count as its last one (i >= n, or directories of a damaged file
        // that promise more ones than the child holds): no read ever leaves the node's arrays
        cnt = cnt < t->nbits ? cnt : t->nbits;
        const uint64_t r1 = ones_before(*t, cnt);
        if (code & 1u) {
            cnt = r1;
            t = &x->nodes[t->right];
        } else {
            cnt -= r1;
            t = &x->nodes[t->left];
        }
        code >>= 1;
    }
    return cnt;
}

// FMIndex::LF(c, i) = C[c] + rank_c(L, i)
__device__ __forceinline__ uint64_t fm_lf(const QIndex *__restrict__ x, uint32_t c, uint64_t i)
{
    const uint64_t base = x->C[c];
    if (x->C[c + 1] == base) return base;
    return base + wt_rank(x, c, i);
}

__global__ void __launch_bounds__(256) search_rank_kernel(const QIndex *__restrict__ x, const uint8_t *__restrict__ c,
                                                          const uint64_t *__restrict__ i, uint64_t *__restrict__ out,
                                                          uint64_t count, int lf)
{
    const uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (q >= count) return;
    out[q] = lf ? fm_lf(x, c[q], i[q]) : wt_rank(x, c[q], i[q]);
}

// HuffWT::access(i, rank): the symbol at position i; *rank = the number of its occurrences in [0, i]
__device__ __forceinline__ uint32_t wt_access(const QIndex *__restrict__ x, uint64_t p, uint64_t &rank)
{
    const QNode *t = &x->nodes[0];
    while (!t->leaf) {
        if (p >= t->nbits) p = t->nbits ? t->nbits - 1 : 0; // never outside the node (see wt_rank)
        const bool bit = (__ldg(t->data + (p >> 6)) >> (p & 63)) & 1u;
        const uint64_t r1 = ones_before(*t, p + 1);
        if (bit) {
            p = r1 - 1;
            t = &x->nodes[t->right];
        } else {
            p = p - r1;
            t = &x->nodes[t->left];
        }
    }
    rank = p + 1;
    return t->ch;
}

__global__ void __launch_bounds__(256) search_access_kernel(const QIndex *__restrict__ x, const uint64_t *__restrict__ i,
                                                            uint8_t *__restrict__ sym, uint64_t *__restrict__ rank,
                                                            uint64_t count)
{
    const uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (q >= count) return;
    uint64_t r;
    sym[q] = (uint8_t)wt_access(x, i[q], r);
    if (rank) rank[q] = r;
}

// Query::pushChar for every symbol of a small alphabet at once (Query.h:37-45; EnumerateQuery.cpp:45-55):
// [sp, ep] -> [LF(c, sp-1), LF(c, ep)-1]; an empty interval (sp > ep) is passed through unchanged.
__global__ void __launch_bounds__(256) search_extend_kernel(const QIndex *__restrict__ x, const uint64_t *__restrict__ sp,
                                                            const uint64_t *__restrict__ ep, uint64_t count,
                                                            const uint8_t *__restrict__ symbols, uint32_t nsym,
                                                            uint64_t *__restrict__ sp_out, uint64_t *__restrict__ ep_out)
{
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (t >= count * nsym) return;
    const uint64_t q = t / nsym;
    const uint32_t c = symbols[t - q * nsym];
    uint64_t lo = sp[q], hi = ep[q];
    if (lo <= hi) {
        lo = fm_lf(x, c, lo - 1);
        hi = fm_lf(x, c, hi) - 1;
    }
    sp_out[t] = lo;
    ep_out[t] = hi;
}

// backward search of whole patterns, last symbol first, from the interval of all suffixes
__global__ void __launch_bounds__(256) search_count_kernel(const QIndex *__restrict__ x, const uint8_t *__restrict__ patterns,
                                                           const uint64_t *__restrict__ offsets, uint64_t count,
                                                           uint64_t *__restrict__ sp_out, uint64_t *__restrict__ ep_out)
{
    const uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (q >= count) return;
    uint64_t lo = 0, hi = x->n - 1;
    for (uint64_t k = offsets[q + 1]; k > offsets[q] && lo <= hi;) {
        const uint32_t c = patterns[--k];
        lo = fm_lf(x, c, lo - 1);
        hi = fm_lf(x, c, hi) - 1;
    }
    sp_out[q] = lo;
    ep_out[q] = hi;
}

// ---- locate / extract over the SA samples of the .sa file (FMIndex::saveSamples, FMIndex.cpp:125-147) --------
// The five sections stay in HBM as the file holds them: BitRank `sampled` (data, Rs, Rb) and the bit-packed
// BlockArrays `suffixes`, `suffixDocId`, `textLength`, `Doc` (fields LSB first, Tools::GetField).  A position is
// resolved by walking LF to the left until the suffix is sampled or starts a document (L[p] = 0).
struct QSamples {
    const uint64_t *data, *Rs; // sampled: one bit per BWT position
    const uint8_t *Rb;
    const uint64_t *suf, *sdoc, *tlen, *doc; // BlockArray words
    uint64_t n;       // BWT length: positions at or behind it are refused
    uint64_t samples; // ones of `sampled` = entries of suf / sdoc (>= 1 whenever a bit is set)
    uint64_t D;       // documents = entries of tlen / doc
    uint64_t maxlen;  // longest document: no walk is longer
    uint32_t wsuf, wdoc, wlen, wend; // field widths of suffixes, suffixDocId, textLength, Doc
    uint32_t *flag;  // kSampleWalk / kSamplePos, read back after every call
};

constexpr uint32_t kSampleWalk = 1; // a walk ran past the longest document: .sa and .fmi do not belong together
constexpr uint32_t kSamplePos = 2;  // a position at or behind n

// Tools::GetField: field i of width len (0..64) of a BlockArray; i < count keeps every read inside its words
__host__ __device__ __forceinline__ uint64_t get_field(const uint64_t *w, uint64_t i, uint32_t len)
{
    if (!len) return 0;
    const uint64_t bit = i * len, k = bit >> 6;
    const uint32_t j = (uint32_t)(bit & 63);
#ifdef __CUDA_ARCH__
    uint64_t v = __ldg(w + k) >> j;
    if (j + len > 64) v |= __ldg(w + k + 1) << (64 - j);
#else
    uint64_t v = w[k] >> j;
    if (j + len > 64) v |= w[k + 1] << (64 - j);
#endif
    return len == 64 ? v : v & ((1ull << len) - 1);
}

// (document, offset) of the suffix at BWT position p; false if the walk does not end within the longest document
__device__ __forceinline__ bool locate_one(const QIndex *__restrict__ x, const QSamples &S, uint64_t p, uint32_t &doc,
                                           uint64_t &off)
{
    for (uint64_t d = 0; d <= S.maxlen; ++d) {
        if (p >= S.n) return false;
        const uint64_t w = __ldg(S.data + (p >> 6));
        if ((w >> (p & 63)) & 1u) {
            // sampled suffix j = rank1(p) - 1 = ones in front of p; the directories come from the file: clamp
            uint64_t j = __ldg(S.Rs + (p >> 8)) + __ldg(S.Rb + (p >> 6)) + (uint64_t)__popcll(w & ((1ull << (p & 63)) - 1));
            j = j < S.samples ? j : S.samples - 1;
            doc = (uint32_t)get_field(S.sdoc, j, S.wdoc);
            off = get_field(S.suf, j, S.wsuf) + d;
            return true;
        }
        uint64_t r;
        const uint32_t c = wt_access(x, p, r);
        if (c == 0) { // the suffix starts a document: the r-th end marker in BWT order names it
            if (!S.D) return false;
            const uint64_t k = r - 1 < S.D ? r - 1 : S.D - 1;
            doc = (uint32_t)get_field(S.doc, k, S.wend);
            off = d;
            return true;
        }
        p = x->C[c] + r - 1; // LF: one text position to the left
    }
    return false;
}

// One thread per position: pos[q], or -- with `starts` -- position q of the intervals [sp[k], sp[k] + starts[k+1] -
// starts[k]) laid end to end (starts: exclusive prefix sums of the interval sizes, starts[nint] = count).
__global__ void __launch_bounds__(256) search_locate_kernel(const QIndex *__restrict__ x, const QSamples S,
                                                            const uint64_t *__restrict__ pos, const uint64_t *__restrict__ sp,
                                                            const uint64_t *__restrict__ starts, uint64_t nint, uint64_t count,
                                                            uint32_t *__restrict__ doc, uint64_t *__restrict__ off)
{
    const uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (q >= count) return;
    uint64_t p;
    if (starts) {
        uint64_t lo = 0, hi = nint - 1; // last k with starts[k] <= q (empty intervals share their start with the next)
        while (lo < hi) {
            const uint64_t mid = (lo + hi + 1) >> 1;
            if (starts[mid] <= q) lo = mid;
            else hi = mid - 1;
        }
        p = sp[lo] + (q - starts[lo]);
    } else {
        p = pos[q];
    }
    uint32_t dk = 0;
    uint64_t o = 0;
    if (p >= S.n) {
        atomicOr(S.flag, kSamplePos);
    } else if (!locate_one(x, S, p, dk, o)) {
        atomicOr(S.flag, kSampleWalk);
    }
    doc[q] = dk;
    off[q] = o;
}

// One thread per document: the terminator suffix of document k sorts at BWT position k; walking LF from there reads
// the document right to left.  out[begin[q] ..) has room for textLength[docs[q]] symbols.
__global__ void __launch_bounds__(256) search_extract_kernel(const QIndex *__restrict__ x, const QSamples S,
                                                             const uint32_t *__restrict__ docs, const uint64_t *__restrict__ begin,
                                                             uint64_t count, uint8_t *__restrict__ out)
{
    const uint64_t q = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (q >= count) return;
    const uint32_t k = docs[q];
    const uint64_t len = get_field(S.tlen, k, S.wlen);
    uint8_t *dst = out + begin[q];
    uint64_t p = k, r, i = len;
    for (; i > 0; --i) {
        const uint32_t c = wt_access(x, p, r);
        if (c == 0) break;
        dst[i - 1] = (uint8_t)c;
        p = x->C[c] + r - 1;
    }
    // the walk must reach the document's start after exactly textLength steps
    if (i || wt_access(x, p, r) != 0) atomicOr(S.flag, kSampleWalk);
}

// ---- the mining client's trie walk, level by level (SURVEY 8 f-4) -----------------------------------------
// EnumerateQuery (EnumerateQuery.cpp:9-58, 151-290) walks the trie of the substrings that occur at least fmin
// times depth-first, one backward-search step per edge, carrying for every node the interval [sp, ep] of the
// pattern and the four intervals of "pattern followed by A / C / G / T" (its left characters, in the orientation
// of the reversed reads).  The same nodes level by level: one thread per (node, symbol) takes the step, the
// surviving children are compacted in order (children of a node stay together, symbols in ACGT order), and every
// node leaves a small record -- frequency, left-character code, symbol, children -- from which the host writes
// the client's byte stream in the reference's depth-first order.
struct EnumNode {
    uint64_t sp, ep;
    uint64_t emin[4], emax[4];
};

__device__ __forceinline__ char enum_left_char(const EnumNode &x)
{
    // EnumerateQuery::leftChar (EnumerateQuery.cpp:77-103)
    bool matches = false, any = false;
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (x.emin[i] <= x.emax[i]) {
            any = true;
            c = i;
            if (x.emin[i] == x.sp && x.emax[i] == x.ep) matches = true;
        }
    }
    const char alphabet[4] = {'A', 'C', 'G', 'T'};
    return matches ? alphabet[c] : (any ? 'N' : '0');
}

// EnumerateQuery::pushChar for symbol c on node x; false if the pattern does not occur
__device__ __forceinline__ bool enum_step(const QIndex *__restrict__ q, const EnumNode &x, uint32_t c, EnumNode &y)
{
    y.sp = fm_lf(q, c, x.sp - 1);
    y.ep = fm_lf(q, c, x.ep) - 1;
    if (y.sp > y.ep) return false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint64_t lo = x.emin[i], hi = x.emax[i];
        if (lo <= hi) {
            lo = fm_lf(q, c, lo - 1);
            hi = fm_lf(q, c, hi) - 1;
        }
        y.emin[i] = lo;
        y.emax[i] = hi;
    }
    return true;
}

// the root and the enforced path (EnumerateQuery::enumerate / nextEnforced): chain[d] = node of path[0..d), d = 0..len;
// *reached = number of path symbols that could be pushed with at least fmin occurrences
__global__ void enum_chain_kernel(const QIndex *__restrict__ q, const uint8_t *__restrict__ path, uint32_t len, uint64_t fmin,
                                  EnumNode *__restrict__ chain, uint32_t *__restrict__ reached)
{
    if (threadIdx.x || blockIdx.x) return;
    const uint8_t alphabet[4] = {'A', 'C', 'G', 'T'};
    EnumNode x;
    x.sp = 0;
    x.ep = q->n - 1;
    for (int i = 0; i < 4; ++i) {
        x.emin[i] = fm_lf(q, alphabet[i], ~0ull);
        x.emax[i] = fm_lf(q, alphabet[i], q->n - 1) - 1;
    }
    chain[0] = x;
    uint32_t d = 0;
    for (; d < len; ++d) {
        EnumNode y;
        if (!enum_step(q, x, path[d], y) || y.ep - y.sp + 1 < fmin) break;
        chain[d + 1] = y;
        x = y;
    }
    *reached = d;
}

// which of the four children of every frontier node survive
__global__ void __launch_bounds__(256) enum_count_kernel(const QIndex *__restrict__ q, const EnumNode *__restrict__ front,
                                                         uint64_t m, uint64_t fmin, uint8_t *__restrict__ mask)
{
    const uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint64_t i = t >> 2;
    const int c = (int)(t & 3);
    bool ok = false;
    if (i < m) {
        const uint8_t alphabet[4] = {'A', 'C', 'G', 'T'};
        const uint64_t sp = fm_lf(q, alphabet[c], front[i].sp - 1), ep = fm_lf(q, alphabet[c], front[i].ep) - 1;
        ok = sp <= ep && ep - sp + 1 >= fmin;
    }
    // the four threads of a node sit in one warp (4 divides 32)
    const uint32_t b = __ballot_sync(0xffffffffu, ok);
    if (i < m && c == 0) mask[i] = (uint8_t)((b >> (threadIdx.x & 28)) & 15u);
}

// per-block sums of the child counts, then (after a scan of the sums) the child offsets and the children
__global__ void __launch_bounds__(256) enum_sum_kernel(const uint8_t *__restrict__ mask, uint64_t m, uint64_t *__restrict__ block_sum)
{
    __shared__ uint32_t s[8];
    const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    uint32_t c = i < m ? __popc(mask[i]) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int k = 0; k < 8; ++k) tot += s[k];
        block_sum[blockIdx.x] = tot;
    }
}

__global__ void __launch_bounds__(1024) enum_scan_kernel(uint64_t *__restrict__ v, uint64_t nblocks)
{
    // exclusive scan in place, total behind the last entry; one block
    __shared__ uint64_t warp_tot[32];
    __shared__ uint64_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint64_t base = 0; base < nblocks; base += 1024) {
        const uint64_t i = base + threadIdx.x;
        const uint64_t x = i < nblocks ? v[i] : 0;
        uint64_t incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
        __syncthreads();
        uint64_t before = carry_s;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += warp_tot[w];
        if (i < nblocks) v[i] = before + incl - x;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) v[nblocks] = carry_s;
}

struct EnumRecord { // what the host needs of a node to write its part of the stream
    uint64_t freq;
    uint64_t child_begin; // index of its first child in the next level
    uint8_t sym, left, mask, pad[5];
};

__global__ void __launch_bounds__(256)
enum_write_kernel(const QIndex *__restrict__ q, const EnumNode *__restrict__ front, uint64_t m, const uint8_t *__restrict__ mask,
                  const uint64_t *__restrict__ block_off, EnumNode *__restrict__ next, EnumRecord *__restrict__ rec_cur,
                  EnumRecord *__restrict__ rec_next)
{
    __shared__ uint32_t s[8];
    const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint32_t mk = i < m ? mask[i] : 0u;
    const uint32_t c = __popc(mk);
    // exclusive prefix of the child counts inside the block
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) s[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t before = incl - c;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += s[w];
    if (i >= m) return;
    uint64_t j = block_off[blockIdx.x] + before;
    rec_cur[i].child_begin = j;
    rec_cur[i].mask = (uint8_t)mk;
    const uint8_t alphabet[4] = {'A', 'C', 'G', 'T'};
    const EnumNode x = front[i];
    for (int k = 0; k < 4; ++k) {
        if (!((mk >> k) & 1u)) continue;
        EnumNode y;
        enum_step(q, x, alphabet[k], y);
        next[j] = y;
        EnumRecord r;
        r.freq = y.ep - y.sp + 1;
        r.child_begin = 0;
        r.sym = alphabet[k];
        r.left = (uint8_t)enum_left_char(y);
        r.mask = 0;
        rec_next[j] = r;
        ++j;
    }
}

std::string g_search_create_error;

} // namespace
} // namespace dsmfm

using namespace dsmfm;

struct dsmfm_searcher {
    int device = 0;
    cudaStream_t stream = nullptr;
    QIndex *d_index = nullptr;
    uint8_t *d_blob = nullptr;
    size_t blob_bytes = 0;
    uint64_t n = 0;
    uint64_t terminators = 0; // C[1] - C[0]: documents of the index
    // SA samples (dsmfm_searcher_load_samples): one device allocation that `samples` points into, and the words of
    // textLength on the host, which size the output of extract
    uint8_t *d_samples = nullptr;
    QSamples samples{};
    std::vector<uint64_t> h_tlen;
    // staging for the host-pointer entry points, grown on demand
    uint8_t *d_stage = nullptr;
    size_t stage_bytes = 0;
    std::string err;

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
    uint8_t *stage(size_t bytes)
    {
        if (bytes > stage_bytes) {
            if (d_stage) cudaFree(d_stage);
            d_stage = nullptr;
            stage_bytes = 0;
            DSM_CUDA(cudaMalloc(&d_stage, bytes));
            stage_bytes = bytes;
        }
        return d_stage;
    }
};

namespace {

size_t up8(size_t x) { return (x + 7) & ~(size_t)7; }

// children of the pre-order node list
int link_nodes(const dsmfm_node *nodes, uint32_t n_nodes, uint32_t &next, QIndex &q)
{
    if (next >= n_nodes || next >= 512) return -1;
    const int me = (int)next++;
    q.nodes[me].leaf = nodes[me].leaf;
    q.nodes[me].ch = nodes[me].ch;
    q.nodes[me].left = q.nodes[me].right = -1;
    q.nodes[me].nbits = nodes[me].leaf ? 0 : nodes[me].nbits;
    if (!nodes[me].leaf) {
        // BitRank.cpp:97-101: integers = ceil((n+1)/64); the kernels index data/Rs/Rb by positions <= nbits
        if (nodes[me].integers != nodes[me].nbits / 64 + 1 || !nodes[me].data || !nodes[me].Rs || !nodes[me].Rb) return -1;
        const int l = link_nodes(nodes, n_nodes, next, q);
        const int r = link_nodes(nodes, n_nodes, next, q);
        if (l < 0 || r < 0) return -1;
        q.nodes[me].left = l;
        q.nodes[me].right = r;
    }
    return me;
}

int searcher_from_index(int device, const dsmfm_index *idx, dsmfm_searcher **out)
{
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_search_create_error = "no CUDA device available (this library has no CPU fallback)";
        return DSMFM_ECUDA;
    }
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev) {
        g_search_create_error = "device ordinal out of range";
        return DSMFM_EINVAL;
    }
    if (!idx || !idx->nodes || idx->n_nodes == 0 || idx->n_nodes > 512) {
        g_search_create_error = "index without a wavelet tree (or with more than 512 nodes)";
        return DSMFM_EINVAL;
    }
    dsmfm_searcher *s = new (std::nothrow) dsmfm_searcher();
    QIndex *q = new (std::nothrow) QIndex();
    if (!s || !q) {
        delete s;
        delete q;
        return DSMFM_ENOMEM;
    }
    std::memset(q, 0, sizeof *q);
    s->device = device;
    s->n = idx->n;
    s->terminators = idx->C[1] - idx->C[0];
    q->n = idx->n;
    std::memcpy(q->C, idx->C, sizeof idx->C);
    q->C[256] = idx->n;
    for (int c = 0; c < 256; ++c) {
        q->code[c] = idx->codetable[c].code;
        q->present[c] = idx->codetable[c].count != 0;
    }
    uint32_t next = 0;
    if (link_nodes(idx->nodes, idx->n_nodes, next, *q) < 0 || next != idx->n_nodes ||
        (!idx->nodes[0].leaf && idx->nodes[0].nbits != idx->n)) {
        g_search_create_error = "malformed wavelet tree";
        delete s;
        delete q;
        return DSMFM_EINVAL;
    }
    size_t total = 0;
    for (uint32_t i = 0; i < idx->n_nodes; ++i) {
        const dsmfm_node &nd = idx->nodes[i];
        if (nd.leaf) continue;
        total += up8(8 * nd.integers) + up8(8 * (nd.nbits / 256 + 1)) + up8(nd.nbits / 64 + 1);
    }
    try {
        DSM_CUDA(cudaSetDevice(device));
        DSM_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        DSM_CUDA(cudaMalloc(&s->d_blob, total ? total : 8));
        s->blob_bytes = total;
        size_t off = 0;
        for (uint32_t i = 0; i < idx->n_nodes; ++i) {
            const dsmfm_node &nd = idx->nodes[i];
            if (nd.leaf) continue;
            const size_t b_data = 8 * nd.integers, b_rs = 8 * (nd.nbits / 256 + 1), b_rb = nd.nbits / 64 + 1;
            DSM_CUDA(cudaMemcpyAsync(s->d_blob + off, nd.data, b_data, cudaMemcpyHostToDevice, s->stream));
            q->nodes[i].data = reinterpret_cast<const uint64_t *>(s->d_blob + off);
            off += up8(b_data);
            DSM_CUDA(cudaMemcpyAsync(s->d_blob + off, nd.Rs, b_rs, cudaMemcpyHostToDevice, s->stream));
            q->nodes[i].Rs = reinterpret_cast<const uint64_t *>(s->d_blob + off);
            off += up8(b_rs);
            DSM_CUDA(cudaMemcpyAsync(s->d_blob + off, nd.Rb, b_rb, cudaMemcpyHostToDevice, s->stream));
            q->nodes[i].Rb = s->d_blob + off;
            off += up8(b_rb);
        }
        DSM_CUDA(cudaMalloc(&s->d_index, sizeof(QIndex)));
        DSM_CUDA(cudaMemcpyAsync(s->d_index, q, sizeof(QIndex), cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
    } catch (const CudaError &e) {
        g_search_create_error = std::string("CUDA error: ") + cudaGetErrorString(e.code);
        if (s->d_blob) cudaFree(s->d_blob);
        if (s->d_index) cudaFree(s->d_index);
        if (s->stream) cudaStreamDestroy(s->stream);
        delete s;
        delete q;
        return e.code == cudaErrorMemoryAllocation ? DSMFM_ENOMEM : DSMFM_ECUDA;
    }
    delete q;
    *out = s;
    return DSMFM_OK;
}

unsigned grid_of(uint64_t threads) { return (unsigned)((threads + 255) / 256); }

#define SEARCH_GUARD(s)                                       \
    if (!(s)) return DSMFM_EINVAL;                            \
    if (cudaSetDevice((s)->device) != cudaSuccess) return (s)->fail(DSMFM_ECUDA, "cudaSetDevice failed")

} // namespace

extern "C" {

DSMFM_API int dsmfm_searcher_create(int device, const dsmfm_index *idx, dsmfm_searcher **out)
{
    if (!out) return DSMFM_EINVAL;
    try {
        return searcher_from_index(device, idx, out);
    } catch (const std::bad_alloc &) {
        g_search_create_error = "host allocation failed";
        return DSMFM_ENOMEM;
    }
}

static int searcher_open_impl(int device, const char *fmi_path, dsmfm_searcher **out);

// FMIndex::FMIndex(FILE *) (FMIndex.cpp:245-357), HuffWT::load (HuffWT.cpp:57-71, 201-207), BitRank::BitRank(FILE *)
// (BitRank.cpp:111-132): only what the queries need -- n, C, the code table and the tree.
DSMFM_API int dsmfm_searcher_open(int device, const char *fmi_path, dsmfm_searcher **out)
{
    if (!out || !fmi_path) return DSMFM_EINVAL;
    *out = nullptr;
    try {
        return searcher_open_impl(device, fmi_path, out);
    } catch (const std::bad_alloc &) { // the whole file and aligned copies of its arrays live in host vectors
        g_search_create_error = "host allocation failed while loading the .fmi file";
        return DSMFM_ENOMEM;
    }
}

static int searcher_open_impl(int device, const char *fmi_path, dsmfm_searcher **out)
{
    FILE *f = std::fopen(fmi_path, "rb");
    if (!f) {
        g_search_create_error = std::string("unable to open ") + fmi_path;
        return DSMFM_EIO;
    }
    std::fseek(f, 0, SEEK_END);
    const long sz = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    std::vector<uint8_t> img((size_t)(sz > 0 ? sz : 0));
    const bool ok = sz > 0 && std::fread(img.data(), 1, (size_t)sz, f) == (size_t)sz;
    std::fclose(f);
    const size_t head = 1 + 8 + 4 + 2048 + 8 + 4096;
    if (!ok || img.size() < head + 2 || img[0] != 17) {
        g_search_create_error = "not a version-17 .fmi file";
        return DSMFM_EINVAL;
    }
    dsmfm_index idx;
    std::memset(&idx, 0, sizeof idx);
    size_t pos = 1;
    std::memcpy(&idx.n, &img[pos], 8); pos += 8;
    std::memcpy(&idx.samplerate, &img[pos], 4); pos += 4;
    std::memcpy(idx.C, &img[pos], 2048); pos += 2048 + 8;
    for (int c = 0; c < 256; ++c) {
        std::memcpy(&idx.codetable[c].count, &img[pos], 8);
        std::memcpy(&idx.codetable[c].bits, &img[pos + 8], 4);
        std::memcpy(&idx.codetable[c].code, &img[pos + 12], 4);
        pos += 16;
    }
    // the arrays sit at odd offsets in the file: aligned copies
    std::vector<dsmfm_node> nodes;
    std::vector<std::vector<uint64_t>> keep;
    int open_children = 1;
    while (open_children > 0) {
        if (pos + 2 > img.size() || nodes.size() >= 512) {
            g_search_create_error = "truncated .fmi file";
            return DSMFM_EINVAL;
        }
        dsmfm_node nd;
        std::memset(&nd, 0, sizeof nd);
        nd.leaf = img[pos++] != 0;
        nd.ch = img[pos++];
        --open_children;
        if (!nd.leaf) {
            uint32_t b = 0, sf = 0;
            if (pos + 24 > img.size()) return DSMFM_EINVAL;
            std::memcpy(&nd.nbits, &img[pos], 8);
            std::memcpy(&nd.integers, &img[pos + 8], 8);
            std::memcpy(&b, &img[pos + 16], 4);
            std::memcpy(&sf, &img[pos + 20], 4);
            pos += 24;
            // sizes come from the file: bound them by the file before any arithmetic can wrap
            const size_t left = img.size() - pos;
            const bool sane = b == 64 && sf == 256 && nd.nbits / 8 <= left && nd.integers == nd.nbits / 64 + 1 &&
                              (nodes.empty() ? nd.nbits == idx.n : nd.nbits <= idx.n);
            const size_t b_data = sane ? 8 * nd.integers : 0, b_rs = sane ? 8 * (nd.nbits / 256 + 1) : 0,
                         b_rb = sane ? nd.nbits / 64 + 1 : 0;
            if (!sane || b_data > left || b_rs > left - b_data || b_rb > left - b_data - b_rs) {
                g_search_create_error = "malformed BitRank in the .fmi file";
                return DSMFM_EINVAL;
            }
            for (size_t bytes : {b_data, b_rs, b_rb}) {
                keep.emplace_back((bytes + 7) / 8 + 1);
                std::memcpy(keep.back().data(), &img[pos], bytes);
                pos += bytes;
            }
            nd.data = keep[keep.size() - 3].data();
            nd.Rs = keep[keep.size() - 2].data();
            nd.Rb = reinterpret_cast<const uint8_t *>(keep[keep.size() - 1].data());
            open_children += 2;
        }
        nodes.push_back(nd);
    }
    idx.n_nodes = (uint32_t)nodes.size();
    idx.nodes = nodes.data();
    return searcher_from_index(device, &idx, out);
}

DSMFM_API uint64_t dsmfm_searcher_length(const dsmfm_searcher *s) { return s ? s->n : 0; }

static int rank_or_lf(dsmfm_searcher *s, const uint8_t *c, const uint64_t *i, uint64_t *out, uint64_t count, int lf,
                      bool on_device)
{
    SEARCH_GUARD(s);
    if (count == 0) return DSMFM_OK;
    if (!c || !i || !out) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        if (on_device) {
            search_rank_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, c, i, out, count, lf);
            DSM_LAUNCH_CHECK();
            DSM_CUDA(cudaStreamSynchronize(s->stream));
            return DSMFM_OK;
        }
        uint8_t *st = s->stage(count * 17 + 64);
        uint64_t *d_i = reinterpret_cast<uint64_t *>(st), *d_o = d_i + count;
        uint8_t *d_c = reinterpret_cast<uint8_t *>(d_o + count);
        DSM_CUDA(cudaMemcpyAsync(d_i, i, count * 8, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemcpyAsync(d_c, c, count, cudaMemcpyHostToDevice, s->stream));
        search_rank_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, d_c, d_i, d_o, count, lf);
        DSM_LAUNCH_CHECK();
        DSM_CUDA(cudaMemcpyAsync(out, d_o, count * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
    } catch (const CudaError &e) {
        return s->fail(DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code, cudaGetErrorString(e.code), e.file, e.line);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_searcher_rank(dsmfm_searcher *s, const uint8_t *c, const uint64_t *i, uint64_t *out, uint64_t count)
{
    return rank_or_lf(s, c, i, out, count, 0, false);
}

DSMFM_API int dsmfm_searcher_lf(dsmfm_searcher *s, const uint8_t *c, const uint64_t *i, uint64_t *out, uint64_t count)
{
    return rank_or_lf(s, c, i, out, count, 1, false);
}

DSMFM_API int dsmfm_searcher_lf_device(dsmfm_searcher *s, const void *c_dev, const void *i_dev, void *out_dev, uint64_t count)
{
    return rank_or_lf(s, static_cast<const uint8_t *>(c_dev), static_cast<const uint64_t *>(i_dev),
                      static_cast<uint64_t *>(out_dev), count, 1, true);
}

DSMFM_API int dsmfm_searcher_access(dsmfm_searcher *s, const uint64_t *i, uint8_t *sym, uint64_t *rank, uint64_t count)
{
    SEARCH_GUARD(s);
    if (count == 0) return DSMFM_OK;
    if (!i || !sym) return s->fail(DSMFM_EINVAL, "null argument");
    for (uint64_t k = 0; k < count; ++k)
        if (i[k] >= s->n) return s->fail(DSMFM_EINVAL, "position %llu is outside the index", (unsigned long long)i[k]);
    try {
        uint8_t *st = s->stage(count * 17 + 64);
        uint64_t *d_i = reinterpret_cast<uint64_t *>(st), *d_r = d_i + count;
        uint8_t *d_s = reinterpret_cast<uint8_t *>(d_r + count);
        DSM_CUDA(cudaMemcpyAsync(d_i, i, count * 8, cudaMemcpyHostToDevice, s->stream));
        search_access_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, d_i, d_s, d_r, count);
        DSM_LAUNCH_CHECK();
        DSM_CUDA(cudaMemcpyAsync(sym, d_s, count, cudaMemcpyDeviceToHost, s->stream));
        if (rank) DSM_CUDA(cudaMemcpyAsync(rank, d_r, count * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
    } catch (const CudaError &e) {
        return s->fail(DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code, cudaGetErrorString(e.code), e.file, e.line);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_searcher_extend(dsmfm_searcher *s, const uint64_t *sp, const uint64_t *ep, uint64_t count,
                                    const uint8_t *symbols, uint32_t nsym, uint64_t *sp_out, uint64_t *ep_out)
{
    SEARCH_GUARD(s);
    if (count == 0 || nsym == 0) return DSMFM_OK;
    if (!sp || !ep || !symbols || !sp_out || !ep_out) return s->fail(DSMFM_EINVAL, "null argument");
    if (nsym > 256) return s->fail(DSMFM_EINVAL, "more than 256 symbols");
    try {
        const uint64_t total = count * nsym;
        uint8_t *st = s->stage(16 * count + 16 * total + 256 + 64);
        uint64_t *d_sp = reinterpret_cast<uint64_t *>(st), *d_ep = d_sp + count, *d_so = d_ep + count, *d_eo = d_so + total;
        uint8_t *d_sym = reinterpret_cast<uint8_t *>(d_eo + total);
        DSM_CUDA(cudaMemcpyAsync(d_sp, sp, count * 8, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemcpyAsync(d_ep, ep, count * 8, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemcpyAsync(d_sym, symbols, nsym, cudaMemcpyHostToDevice, s->stream));
        search_extend_kernel<<<grid_of(total), 256, 0, s->stream>>>(s->d_index, d_sp, d_ep, count, d_sym, nsym, d_so, d_eo);
        DSM_LAUNCH_CHECK();
        DSM_CUDA(cudaMemcpyAsync(sp_out, d_so, total * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaMemcpyAsync(ep_out, d_eo, total * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
    } catch (const CudaError &e) {
        return s->fail(DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code, cudaGetErrorString(e.code), e.file, e.line);
    }
    return DSMFM_OK;
}

DSMFM_API int dsmfm_searcher_count(dsmfm_searcher *s, const uint8_t *patterns, const uint64_t *offsets, uint64_t count,
                                   uint64_t *sp_out, uint64_t *ep_out)
{
    SEARCH_GUARD(s);
    if (count == 0) return DSMFM_OK;
    if (!patterns || !offsets || !sp_out || !ep_out) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        const uint64_t bytes = offsets[count];
        uint8_t *st = s->stage(8 * (count + 1) + 16 * count + bytes + 64);
        uint64_t *d_off = reinterpret_cast<uint64_t *>(st), *d_so = d_off + count + 1, *d_eo = d_so + count;
        uint8_t *d_pat = reinterpret_cast<uint8_t *>(d_eo + count);
        DSM_CUDA(cudaMemcpyAsync(d_off, offsets, (count + 1) * 8, cudaMemcpyHostToDevice, s->stream));
        if (bytes) DSM_CUDA(cudaMemcpyAsync(d_pat, patterns, bytes, cudaMemcpyHostToDevice, s->stream));
        search_count_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, d_pat, d_off, count, d_so, d_eo);
        DSM_LAUNCH_CHECK();
        DSM_CUDA(cudaMemcpyAsync(sp_out, d_so, count * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaMemcpyAsync(ep_out, d_eo, count * 8, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
    } catch (const CudaError &e) {
        return s->fail(DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code, cudaGetErrorString(e.code), e.file, e.line);
    }
    return DSMFM_OK;
}

// ---- locate / extract over the SA samples (FMIndex::loadSamples, FMIndex::locate / getSuffix) -------------------
namespace {

// The .sa layout FMIndex::saveSamples writes (FMIndex.cpp:134-143; dsmfm_sa_serialize): BitRank `sampled` (BitRank::save:
// n, integers, 64, 256, data[integers], Rs[n/256+1], Rb[n/64+1]), then the BlockArrays suffixes, suffixDocId,
// textLength, Doc (BlockArray::Save: count, width, words[count*width/64+1]).  Everything is checked against this index
// before anything is uploaded; the samples attached before stay in place if the image is refused.
int samples_set_impl(dsmfm_searcher *s, const uint8_t *img, uint64_t bytes)
{
    auto bad = [&](const char *what) { return s->fail(DSMFM_EINVAL, "SA samples: %s", what); };
    uint64_t pos = 0;
    auto left = [&]() { return bytes - pos; };
    auto u64 = [&](uint64_t at) { uint64_t v; std::memcpy(&v, img + at, 8); return v; };
    if (bytes < 24) return bad("truncated header of `sampled`");
    const uint64_t n = u64(0), integers = u64(8);
    uint32_t b, sf;
    std::memcpy(&b, img + 16, 4);
    std::memcpy(&sf, img + 20, 4);
    pos = 24;
    if (n != s->n)
        return s->fail(DSMFM_EINVAL, "SA samples of an index of %llu symbols, this index has %llu", (unsigned long long)n,
                       (unsigned long long)s->n);
    if (integers != n / 64 + 1 || b != 64 || sf != 256) return bad("malformed BitRank `sampled`");
    // n is this index's length, so none of these sizes can wrap
    const uint64_t b_data = 8 * integers, b_rs = 8 * (n / 256 + 1), b_rb = n / 64 + 1;
    if (b_data > left() || b_rs > left() - b_data || b_rb > left() - b_data - b_rs) return bad("truncated `sampled`");
    const uint64_t o_data = pos, o_rs = o_data + b_data, o_rb = o_rs + b_rs;
    pos = o_rb + b_rb;
    uint64_t ones = 0; // among the first n bits: the kernels never look behind them
    for (uint64_t w = 0; w <= n / 64; ++w) {
        uint64_t x = u64(o_data + 8 * w);
        if (w == n / 64) x &= (1ull << (n & 63)) - 1;
        ones += (uint64_t)__builtin_popcountll(x);
    }
    struct Arr {
        uint64_t count, width, off, words;
    } a[4];
    for (Arr &x : a) {
        if (left() < 16) return bad("truncated BlockArray header");
        x.count = u64(pos);
        x.width = u64(pos + 8);
        pos += 16;
        if (x.count > n || x.width > 64) return bad("malformed BlockArray header");
        x.words = x.count * x.width / 64 + 1;
        if (x.words > left() / 8) return bad("truncated BlockArray");
        x.off = pos;
        pos += 8 * x.words;
    }
    if (pos != bytes) return s->fail(DSMFM_EINVAL, "SA samples: %llu bytes behind the last section", (unsigned long long)left());
    const Arr &suf = a[0], &sdoc = a[1], &tlen = a[2], &doc = a[3];
    if (sdoc.width > 32 || doc.width > 32) return bad("document ids wider than 32 bits");
    if (suf.count != ones || sdoc.count != ones)
        return s->fail(DSMFM_EINVAL, "SA samples: %llu / %llu samples for %llu sampled positions", (unsigned long long)suf.count,
                       (unsigned long long)sdoc.count, (unsigned long long)ones);
    const uint64_t D = s->terminators;
    if (tlen.count != D || doc.count != D)
        return s->fail(DSMFM_EINVAL, "SA samples: %llu / %llu document entries, the index has %llu documents",
                       (unsigned long long)tlen.count, (unsigned long long)doc.count, (unsigned long long)D);
    auto words_of = [&](const Arr &x) {
        std::vector<uint64_t> v(x.words);
        std::memcpy(v.data(), img + x.off, 8 * x.words);
        return v;
    };
    std::vector<uint64_t> w_tlen = words_of(tlen);
    uint64_t sum = 0, maxlen = 0;
    for (uint64_t k = 0; k < D; ++k) {
        const uint64_t t = get_field(w_tlen.data(), k, (uint32_t)tlen.width);
        if (t > n - sum) return bad("document lengths add up to more than the index"); // (sum <= n: cannot wrap)
        sum += t;
        maxlen = t > maxlen ? t : maxlen;
    }
    if (sum + D != n)
        return s->fail(DSMFM_EINVAL, "SA samples: document lengths add up to %llu + %llu terminators, the index has %llu symbols",
                       (unsigned long long)sum, (unsigned long long)D, (unsigned long long)n);
    for (const Arr *x : {&sdoc, &doc}) {
        const std::vector<uint64_t> w = words_of(*x);
        for (uint64_t j = 0; j < x->count; ++j)
            if (get_field(w.data(), j, (uint32_t)x->width) >= D) return bad("document id out of range");
    }

    uint8_t *blob = nullptr;
    try {
        // flag word, then the sections in file order, each at an 8-byte boundary
        const uint64_t sizes[7] = {b_data, b_rs, b_rb, 8 * suf.words, 8 * sdoc.words, 8 * tlen.words, 8 * doc.words};
        const uint64_t from[7] = {o_data, o_rs, o_rb, suf.off, sdoc.off, tlen.off, doc.off};
        uint64_t at[7], total = 8;
        for (int i = 0; i < 7; ++i) {
            at[i] = total;
            total += up8(sizes[i]);
        }
        DSM_CUDA(cudaMalloc(&blob, total));
        DSM_CUDA(cudaMemsetAsync(blob, 0, 8, s->stream));
        for (int i = 0; i < 7; ++i)
            DSM_CUDA(cudaMemcpyAsync(blob + at[i], img + from[i], sizes[i], cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaStreamSynchronize(s->stream));
        QSamples &S = s->samples;
        S.data = reinterpret_cast<const uint64_t *>(blob + at[0]);
        S.Rs = reinterpret_cast<const uint64_t *>(blob + at[1]);
        S.Rb = blob + at[2];
        S.suf = reinterpret_cast<const uint64_t *>(blob + at[3]);
        S.sdoc = reinterpret_cast<const uint64_t *>(blob + at[4]);
        S.tlen = reinterpret_cast<const uint64_t *>(blob + at[5]);
        S.doc = reinterpret_cast<const uint64_t *>(blob + at[6]);
        S.n = n;
        S.samples = ones;
        S.D = D;
        S.maxlen = maxlen;
        S.wsuf = (uint32_t)suf.width;
        S.wdoc = (uint32_t)sdoc.width;
        S.wlen = (uint32_t)tlen.width;
        S.wend = (uint32_t)doc.width;
        S.flag = reinterpret_cast<uint32_t *>(blob);
    } catch (const CudaError &e) {
        if (blob) cudaFree(blob);
        return s->fail(e.code == cudaErrorMemoryAllocation ? DSMFM_ENOMEM : DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d",
                       (int)e.code, cudaGetErrorString(e.code), e.file, e.line);
    }
    if (s->d_samples) cudaFree(s->d_samples);
    s->d_samples = blob;
    s->h_tlen.swap(w_tlen);
    return DSMFM_OK;
}

#define SAMPLES_GUARD(s)                                                                                    \
    SEARCH_GUARD(s);                                                                                        \
    if (!(s)->d_samples) return (s)->fail(DSMFM_EINVAL, "no SA samples attached (dsmfm_searcher_load_samples)")

// the flag the walks raise; the stream has been synchronised by the caller's copies
int samples_verdict(dsmfm_searcher *s)
{
    uint32_t f = 0;
    DSM_CUDA(cudaMemcpyAsync(&f, s->samples.flag, 4, cudaMemcpyDeviceToHost, s->stream));
    DSM_CUDA(cudaStreamSynchronize(s->stream));
    if (f & kSamplePos) return s->fail(DSMFM_EINVAL, "locate: position outside the index (n = %llu)", (unsigned long long)s->n);
    if (f & kSampleWalk)
        return s->fail(DSMFM_EINVAL, "SA samples: a walk ran past the longest document (%llu symbols): the .sa file does not "
                                     "belong to this index", (unsigned long long)s->samples.maxlen);
    return DSMFM_OK;
}

void launch_locate(dsmfm_searcher *s, const uint64_t *d_pos, const uint64_t *d_sp, const uint64_t *d_starts, uint64_t nint,
                   uint64_t count, uint32_t *d_doc, uint64_t *d_off)
{
    DSM_CUDA(cudaMemsetAsync(s->samples.flag, 0, 4, s->stream));
    search_locate_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, s->samples, d_pos, d_sp, d_starts, nint, count, d_doc,
                                                                 d_off);
    DSM_LAUNCH_CHECK();
}

int cuda_failure(dsmfm_searcher *s, const CudaError &e)
{
    return s->fail(e.code == cudaErrorMemoryAllocation ? DSMFM_ENOMEM : DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code,
                   cudaGetErrorString(e.code), e.file, e.line);
}

} // namespace

DSMFM_API int dsmfm_searcher_set_samples(dsmfm_searcher *s, const uint8_t *image, uint64_t bytes)
{
    SEARCH_GUARD(s);
    if (!image && bytes) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        return samples_set_impl(s, image, bytes);
    } catch (const std::bad_alloc &) {
        return s->fail(DSMFM_ENOMEM, "host allocation failed");
    }
}

DSMFM_API int dsmfm_searcher_load_samples(dsmfm_searcher *s, const char *sa_path)
{
    SEARCH_GUARD(s);
    if (!sa_path) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        FILE *f = std::fopen(sa_path, "rb");
        if (!f) return s->fail(DSMFM_EIO, "unable to open %s", sa_path);
        std::fseek(f, 0, SEEK_END);
        const long sz = std::ftell(f);
        std::fseek(f, 0, SEEK_SET);
        std::vector<uint8_t> img((size_t)(sz > 0 ? sz : 0));
        const bool ok = sz >= 0 && std::fread(img.data(), 1, img.size(), f) == img.size();
        std::fclose(f);
        if (!ok) return s->fail(DSMFM_EIO, "unable to read %s", sa_path);
        return samples_set_impl(s, img.data(), img.size());
    } catch (const std::bad_alloc &) {
        return s->fail(DSMFM_ENOMEM, "host allocation failed while loading the .sa file");
    }
}

DSMFM_API int dsmfm_searcher_locate(dsmfm_searcher *s, const uint64_t *pos, uint64_t count, uint32_t *doc, uint64_t *offset)
{
    SAMPLES_GUARD(s);
    if (count == 0) return DSMFM_OK;
    if (!pos || !doc || !offset) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        uint8_t *st = s->stage(count * 20 + 64);
        uint64_t *d_pos = reinterpret_cast<uint64_t *>(st), *d_off = d_pos + count;
        uint32_t *d_doc = reinterpret_cast<uint32_t *>(d_off + count);
        DSM_CUDA(cudaMemcpyAsync(d_pos, pos, count * 8, cudaMemcpyHostToDevice, s->stream));
        launch_locate(s, d_pos, nullptr, nullptr, 0, count, d_doc, d_off);
        DSM_CUDA(cudaMemcpyAsync(doc, d_doc, count * 4, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaMemcpyAsync(offset, d_off, count * 8, cudaMemcpyDeviceToHost, s->stream));
        return samples_verdict(s);
    } catch (const CudaError &e) {
        return cuda_failure(s, e);
    }
}

DSMFM_API int dsmfm_searcher_locate_device(dsmfm_searcher *s, const void *pos_dev, uint64_t count, void *doc_dev, void *offset_dev)
{
    SAMPLES_GUARD(s);
    if (count == 0) return DSMFM_OK;
    if (!pos_dev || !doc_dev || !offset_dev) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        launch_locate(s, static_cast<const uint64_t *>(pos_dev), nullptr, nullptr, 0, count, static_cast<uint32_t *>(doc_dev),
                      static_cast<uint64_t *>(offset_dev));
        return samples_verdict(s);
    } catch (const CudaError &e) {
        return cuda_failure(s, e);
    }
}

DSMFM_API int dsmfm_searcher_locate_ranges(dsmfm_searcher *s, const uint64_t *sp, const uint64_t *ep, uint64_t count,
                                           uint64_t cap, uint32_t *doc, uint64_t *offset, uint64_t *total)
{
    SAMPLES_GUARD(s);
    if (!total || (count && (!sp || !ep))) return s->fail(DSMFM_EINVAL, "null argument");
    *total = 0;
    try {
        std::vector<uint64_t> starts(count + 1);
        uint64_t sum = 0;
        for (uint64_t k = 0; k < count; ++k) {
            starts[k] = sum;
            if (sp[k] > ep[k]) continue;
            if (ep[k] >= s->n)
                return s->fail(DSMFM_EINVAL, "locate_ranges: interval %llu ends at %llu, outside the index", (unsigned long long)k,
                               (unsigned long long)ep[k]);
            sum += ep[k] - sp[k] + 1;
        }
        starts[count] = sum;
        *total = sum;
        if (sum > cap)
            return s->fail(DSMFM_ELIMIT, "locate_ranges: %llu occurrences, room for %llu", (unsigned long long)sum,
                           (unsigned long long)cap);
        if (sum == 0) return DSMFM_OK;
        if (!doc || !offset) return s->fail(DSMFM_EINVAL, "null argument");
        uint8_t *st = s->stage(16 * count + 8 + 12 * sum + 64);
        uint64_t *d_sp = reinterpret_cast<uint64_t *>(st), *d_starts = d_sp + count, *d_off = d_starts + count + 1;
        uint32_t *d_doc = reinterpret_cast<uint32_t *>(d_off + sum);
        DSM_CUDA(cudaMemcpyAsync(d_sp, sp, count * 8, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemcpyAsync(d_starts, starts.data(), (count + 1) * 8, cudaMemcpyHostToDevice, s->stream));
        launch_locate(s, nullptr, d_sp, d_starts, count, sum, d_doc, d_off);
        DSM_CUDA(cudaMemcpyAsync(doc, d_doc, sum * 4, cudaMemcpyDeviceToHost, s->stream));
        DSM_CUDA(cudaMemcpyAsync(offset, d_off, sum * 8, cudaMemcpyDeviceToHost, s->stream));
        return samples_verdict(s);
    } catch (const CudaError &e) {
        return cuda_failure(s, e);
    } catch (const std::bad_alloc &) {
        return s->fail(DSMFM_ENOMEM, "host allocation failed");
    }
}

DSMFM_API int dsmfm_searcher_extract(dsmfm_searcher *s, const uint32_t *docs, uint64_t count, uint8_t *out, uint64_t cap,
                                     uint64_t *offsets)
{
    SAMPLES_GUARD(s);
    if (!offsets || (count && !docs)) return s->fail(DSMFM_EINVAL, "null argument");
    const QSamples &S = s->samples;
    offsets[0] = 0;
    for (uint64_t k = 0; k < count; ++k) {
        if (docs[k] >= S.D)
            return s->fail(DSMFM_EINVAL, "extract: document %u of %llu", docs[k], (unsigned long long)S.D);
        offsets[k + 1] = offsets[k] + get_field(s->h_tlen.data(), docs[k], S.wlen);
    }
    const uint64_t bytes = offsets[count];
    if (bytes > cap)
        return s->fail(DSMFM_ELIMIT, "extract: %llu bytes, room for %llu", (unsigned long long)bytes, (unsigned long long)cap);
    if (count == 0) return DSMFM_OK;
    if (bytes && !out) return s->fail(DSMFM_EINVAL, "null argument");
    try {
        uint8_t *st = s->stage(8 * (count + 1) + 4 * count + bytes + 64);
        uint64_t *d_begin = reinterpret_cast<uint64_t *>(st);
        uint32_t *d_docs = reinterpret_cast<uint32_t *>(d_begin + count + 1);
        uint8_t *d_out = reinterpret_cast<uint8_t *>(d_docs + count);
        DSM_CUDA(cudaMemcpyAsync(d_begin, offsets, (count + 1) * 8, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemcpyAsync(d_docs, docs, count * 4, cudaMemcpyHostToDevice, s->stream));
        DSM_CUDA(cudaMemsetAsync(S.flag, 0, 4, s->stream));
        search_extract_kernel<<<grid_of(count), 256, 0, s->stream>>>(s->d_index, S, d_docs, d_begin, count, d_out);
        DSM_LAUNCH_CHECK();
        if (bytes) DSM_CUDA(cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, s->stream));
        return samples_verdict(s);
    } catch (const CudaError &e) {
        return cuda_failure(s, e);
    }
}

// ---- EnumerateQuery::enumerate as a byte stream -----------------------------------------------------------
namespace {
struct StreamSink {
    int fd = -1;
    std::vector<uint8_t> *mem = nullptr;
    std::vector<uint8_t> buf;
    uint64_t total = 0;
    bool ok = true;
    void flush()
    {
        if (fd >= 0 && ok) {
            size_t done = 0;
            while (done < buf.size()) {
                const ssize_t w = ::write(fd, buf.data() + done, buf.size() - done);
                if (w <= 0) { ok = false; break; }
                done += (size_t)w;
            }
        } else if (mem) {
            mem->insert(mem->end(), buf.begin(), buf.end());
        }
        total += buf.size();
        buf.clear();
    }
    void putc(uint8_t c)
    {
        buf.push_back(c);
        if (buf.size() >= (1u << 20)) flush();
    }
    void putulong(uint64_t u) // ClientSocket::putulong (ClientSocket.h:20-39)
    {
        if (u < 128) { putc((uint8_t)(u | 128u)); return; }
        uint8_t l = 0;
        for (uint64_t t = u; t; t >>= 8) ++l;
        putc(l);
        for (; u; u >>= 8) putc((uint8_t)(u & 0xff));
    }
};

int enumerate_impl(dsmfm_searcher *s, const uint8_t *path, uint32_t path_len, uint64_t fmin, uint32_t maxdepth, StreamSink &out)
{
    SEARCH_GUARD(s);
    if (fmin < 2) return s->fail(DSMFM_EINVAL, "dsmfm_searcher_enumerate: fmin must be at least 2 (fmin 1 walks unary paths one getL at a time)");
    if (path_len && !path) return s->fail(DSMFM_EINVAL, "null path");
    if (s->n < 2) return s->fail(DSMFM_EINVAL, "dsmfm_searcher_enumerate: index of fewer than two symbols");
    cudaStream_t st = s->stream;
    std::vector<std::vector<EnumRecord>> levels; // levels[0] = the node at the end of the enforced path (or the root)
    std::vector<EnumNode> chain(path_len + 1);
    uint32_t reached = 0;
    EnumNode *d_front = nullptr, *d_next = nullptr;
    EnumRecord *d_rec_cur = nullptr, *d_rec_next = nullptr;
    uint8_t *d_mask = nullptr, *d_path = nullptr;
    uint64_t *d_block = nullptr;
    uint32_t *d_reached = nullptr;
    auto release = [&]() {
        cudaFree(d_front); cudaFree(d_next); cudaFree(d_rec_cur); cudaFree(d_rec_next); cudaFree(d_mask); cudaFree(d_path);
        cudaFree(d_block); cudaFree(d_reached);
    };
    try {
        DSM_CUDA(cudaMalloc(&d_front, sizeof(EnumNode) * (path_len + 1)));
        DSM_CUDA(cudaMalloc(&d_path, path_len + 1));
        DSM_CUDA(cudaMalloc(&d_reached, 4));
        if (path_len) DSM_CUDA(cudaMemcpyAsync(d_path, path, path_len, cudaMemcpyHostToDevice, st));
        enum_chain_kernel<<<1, 32, 0, st>>>(s->d_index, d_path, path_len, fmin, d_front, d_reached);
        DSM_LAUNCH_CHECK();
        DSM_CUDA(cudaMemcpyAsync(chain.data(), d_front, sizeof(EnumNode) * (path_len + 1), cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaMemcpyAsync(&reached, d_reached, 4, cudaMemcpyDeviceToHost, st));
        DSM_CUDA(cudaStreamSynchronize(st));
        cudaFree(d_front);
        d_front = nullptr;
        // the subtree below the enforced path exists only if the whole path could be pushed
        // (depth of its root = path_len; EnumerateQuery::nextSymbol returns at once at maxdepth)
        if (reached == path_len) {
            uint64_t m = 1;
            DSM_CUDA(cudaMalloc(&d_front, sizeof(EnumNode)));
            DSM_CUDA(cudaMemcpyAsync(d_front, &chain[path_len], sizeof(EnumNode), cudaMemcpyHostToDevice, st));
            DSM_CUDA(cudaMalloc(&d_rec_cur, sizeof(EnumRecord)));
            DSM_CUDA(cudaMemsetAsync(d_rec_cur, 0, sizeof(EnumRecord), st));
            uint32_t depth = path_len;
            while (m > 0) {
                levels.emplace_back(m);
                uint64_t next_m = 0;
                if (depth < maxdepth) {
                    const uint64_t nblocks = (m + 255) / 256;
                    DSM_CUDA(cudaMalloc(&d_mask, m));
                    DSM_CUDA(cudaMalloc(&d_block, sizeof(uint64_t) * (nblocks + 1)));
                    enum_count_kernel<<<(unsigned)((4 * m + 255) / 256), 256, 0, st>>>(s->d_index, d_front, m, fmin, d_mask);
                    enum_sum_kernel<<<(unsigned)nblocks, 256, 0, st>>>(d_mask, m, d_block);
                    enum_scan_kernel<<<1, 1024, 0, st>>>(d_block, nblocks);
                    DSM_LAUNCH_CHECK();
                    DSM_CUDA(cudaMemcpyAsync(&next_m, d_block + nblocks, 8, cudaMemcpyDeviceToHost, st));
                    DSM_CUDA(cudaStreamSynchronize(st));
                    DSM_CUDA(cudaMalloc(&d_next, sizeof(EnumNode) * (next_m ? next_m : 1)));
                    DSM_CUDA(cudaMalloc(&d_rec_next, sizeof(EnumRecord) * (next_m ? next_m : 1)));
                    enum_write_kernel<<<(unsigned)nblocks, 256, 0, st>>>(s->d_index, d_front, m, d_mask, d_block, d_next, d_rec_cur,
                                                                          d_rec_next);
                    DSM_LAUNCH_CHECK();
                }
                DSM_CUDA(cudaMemcpyAsync(levels.back().data(), d_rec_cur, sizeof(EnumRecord) * m, cudaMemcpyDeviceToHost, st));
                DSM_CUDA(cudaStreamSynchronize(st));
                cudaFree(d_front); cudaFree(d_rec_cur); cudaFree(d_mask); cudaFree(d_block);
                d_front = d_next;
                d_rec_cur = d_rec_next;
                d_next = nullptr; d_rec_next = nullptr; d_mask = nullptr; d_block = nullptr;
                m = next_m;
                ++depth;
            }
        }
    } catch (const CudaError &e) {
        release();
        return s->fail(e.code == cudaErrorMemoryAllocation ? DSMFM_ENOMEM : DSMFM_ECUDA, "CUDA error %d (%s) at %s:%d", (int)e.code,
                       cudaGetErrorString(e.code), e.file, e.line);
    }
    release();

    // ---- the stream, depth first (EnumerateQuery.cpp:207-222, 273-288) ----
    uint64_t reported = 0;
    auto close_node = [&](uint64_t freq, uint32_t depth, uint8_t left) {
        out.putulong(freq);
        if (depth <= 6) {
            out.putc('R');
            out.putulong(reported);
        }
        out.putc(left);
        out.putc(')');
    };
    auto left_of = [](const EnumNode &x) -> uint8_t {
        bool matches = false, any = false;
        int c = 0;
        for (int i = 0; i < 4; ++i)
            if (x.emin[i] <= x.emax[i]) {
                any = true;
                c = i;
                if (x.emin[i] == x.sp && x.emax[i] == x.ep) matches = true;
            }
        return matches ? (uint8_t)"ACGT"[c] : (any ? 'N' : '0');
    };
    for (uint32_t d = 1; d <= reached; ++d) { // the enforced path opens ...
        out.putc('(');
        out.putc(path[d - 1]);
        ++reported;
    }
    if (reached == path_len && !levels.empty()) {
        // children of the path's last node, depth first with an explicit stack
        struct Frame { uint32_t level; uint64_t idx; uint8_t next; };
        std::vector<Frame> stack;
        auto open_children = [&](uint32_t level, uint64_t idx) { stack.push_back(Frame{level, idx, 0}); };
        open_children(0, 0);
        while (!stack.empty()) {
            Frame &f = stack.back();
            const EnumRecord &r = levels[f.level][f.idx];
            const uint32_t nchild = (uint32_t)__builtin_popcount(r.mask);
            if (f.next < nchild) {
                const uint64_t child = r.child_begin + f.next;
                ++f.next;
                const EnumRecord &c = levels[f.level + 1][child];
                out.putc('(');
                out.putc(c.sym);
                ++reported;
                open_children(f.level + 1, child);
            } else {
                const uint32_t level = f.level;
                const uint64_t idx = f.idx;
                stack.pop_back();
                if (level > 0) { // (level 0 is the path's last node or the root: closed below)
                    const EnumRecord &me = levels[level][idx];
                    close_node(me.freq, path_len + level, me.left);
                }
            }
        }
    }
    for (uint32_t d = reached; d >= 1; --d) // ... and closes, innermost first
        close_node(chain[d].ep - chain[d].sp + 1, d, left_of(chain[d]));
    out.flush();
    if (!out.ok) return s->fail(DSMFM_EIO, "dsmfm_searcher_enumerate: write error");
    return DSMFM_OK;
}
} // namespace

DSMFM_API int dsmfm_searcher_enumerate_fd(dsmfm_searcher *s, const char *enforce_path, uint64_t fmin, uint32_t maxdepth, int fd,
                                          uint64_t *bytes_written)
{
    if (!s) return DSMFM_EINVAL;
    try {
        StreamSink sink;
        sink.fd = fd;
        const size_t len = enforce_path ? std::strlen(enforce_path) : 0;
        const int rc = enumerate_impl(s, reinterpret_cast<const uint8_t *>(enforce_path), (uint32_t)len, fmin, maxdepth ? maxdepth : ~0u, sink);
        if (bytes_written) *bytes_written = sink.total;
        return rc;
    } catch (const std::bad_alloc &) {
        return s->fail(DSMFM_ENOMEM, "host allocation failed");
    }
}

DSMFM_API int dsmfm_searcher_enumerate(dsmfm_searcher *s, const char *enforce_path, uint64_t fmin, uint32_t maxdepth, uint8_t **out,
                                       uint64_t *out_bytes)
{
    if (!s || !out || !out_bytes) return DSMFM_EINVAL;
    *out = nullptr;
    *out_bytes = 0;
    try {
        std::vector<uint8_t> mem;
        StreamSink sink;
        sink.mem = &mem;
        const size_t len = enforce_path ? std::strlen(enforce_path) : 0;
        const int rc = enumerate_impl(s, reinterpret_cast<const uint8_t *>(enforce_path), (uint32_t)len, fmin, maxdepth ? maxdepth : ~0u, sink);
        if (rc) return rc;
        uint8_t *p = static_cast<uint8_t *>(std::malloc(mem.size() ? mem.size() : 1));
        if (!p) return s->fail(DSMFM_ENOMEM, "host allocation failed");
        std::memcpy(p, mem.data(), mem.size());
        *out = p;
        *out_bytes = mem.size();
        return DSMFM_OK;
    } catch (const std::bad_alloc &) {
        return s->fail(DSMFM_ENOMEM, "host allocation failed");
    }
}

DSMFM_API void dsmfm_stream_free(uint8_t *p) { std::free(p); }

DSMFM_API const char *dsmfm_searcher_last_error(const dsmfm_searcher *s)
{
    return s ? s->err.c_str() : g_search_create_error.c_str();
}

DSMFM_API void dsmfm_searcher_destroy(dsmfm_searcher *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->d_samples) cudaFree(s->d_samples);
    if (s->d_stage) cudaFree(s->d_stage);
    if (s->d_blob) cudaFree(s->d_blob);
    if (s->d_index) cudaFree(s->d_index);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

} // extern "C"
