// kernels.cuh -- launch wrappers of the FM-index build kernels (sm_100a).
// Every wrapper enqueues on `stream`, checks the launch and bumps *launches.
#pragma once
#include "common.cuh"

namespace dsmfm {

// ---- ingest -----------------------------------------------------------------
// 256-bin histogram of the raw text (counts[0] = number of documents).
void launch_byte_hist(cudaStream_t st, const uint8_t *raw, uint64_t n, uint64_t *counts, uint32_t *launches);

// Per-chunk terminator summary used to get numberOfTexts / maxTextLength / empty
// documents for bulk-appended text (TextCollectionBuilder.cpp:73-91).
constexpr int kStatChunk = 16384;
struct ChunkStat {
    int64_t first;   // position of the first terminator in the chunk, -1 if none
    int64_t last;    // position of the last terminator in the chunk
    uint64_t maxgap; // largest distance between consecutive terminators inside the chunk
    uint64_t mingap; // smallest such distance (UINT64_MAX if fewer than two)
};
void launch_doc_stats(cudaStream_t st, const uint8_t *raw, uint64_t n, ChunkStat *out, uint32_t *launches);

// raw bytes -> dense codes packed BITS per symbol (common.cuh); `code_map` is a
// device table of 256 bytes.  `nwords` words are written (tail zero-padded).
void launch_pack(cudaStream_t st, int bits, const uint8_t *raw, uint64_t n, const uint8_t *code_map, uint64_t *packed,
                 uint64_t nwords, uint32_t *launches);

// ---- suffix sorting ---------------------------------------------------------
// key[p] = the first `first_syms` (<= SPW) symbols of suffix p, cut at its terminator, right-aligned.
// With carry_prev the code of the symbol before the suffix rides in the BITS bits above the key.
// Also, in ghist[pass][256] (zeroed u64), the counts of the keys' 8-bit digits from bit 0 up to
// first_syms*bits -- the histogram the LSD sort needs (radix_sort_pairs with hist_ready).
// word_begin / word_end (0 = all): only the suffixes starting in these words of the packed text -- a text that
// streams in from the host is keyed piece by piece; the word behind the last one must already be packed.
void launch_make_keys_hist(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n, uint64_t *keys, int first_syms,
                           bool carry_prev, uint64_t *ghist, uint32_t *launches, uint64_t word_begin = 0,
                           uint64_t word_end = 0);

// Group heads after the initial sort: bit i set iff suffix i starts a new group
// (key differs from its predecessor) or is already finished (key holds the
// terminator).  Bits >= n are set.  *remaining += suffixes left in groups of >= 2.
// ---- key-range sharding (multi-GPU) -------------------------------------------
// hist[4096]: counts of the top `top_bits` (<= 12) bits of every suffix's first key
void launch_key_top_hist(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n, int first_syms, int top_bits,
                         unsigned long long *hist, uint32_t *launches);
// (key, position) pairs of the suffixes whose first key lies in [key_lo, key_hi), in text order.  The bounds
// are multiples of 2^(key_bits - top_bits) (bin boundaries of the histogram above).  tile_scratch holds
// select_tiles(...) u64, counter one u32, lut_scratch kSelLutWords u32 (device).
// The packed text may be a row of equally sized SLOTS, one per block of documents (the blocks of the GPUs of a
// multi-GPU build, packed where they lived and exchanged as words): slot s holds geom.bytes[s] symbols from its
// first word on, zero padding behind them.  Positions are positions in this padded ("virtual") text; padding
// positions are never selected.  One block: world = 1, slot_words = all words, bytes[0] = n.
constexpr int kMaxBlocks = 64;
constexpr int kSelLutWords = 2048;
struct SelGeom {
    uint64_t slot_words;
    uint32_t world;
    uint32_t reserved;
    uint64_t bytes[kMaxBlocks];
};
uint64_t select_tiles(uint64_t nwords, int bits, int first_syms, int top_bits);
void launch_select(cudaStream_t st, int bits, const uint64_t *packed, uint64_t nwords, int first_syms, int top_bits,
                   bool carry_prev, uint64_t key_lo, uint64_t key_hi, uint64_t *tile_scratch, uint32_t *counter,
                   uint64_t *keys, uint32_t *vals, int lo_bits, int hi_shift, const SelGeom &geom, uint32_t *lut_scratch,
                   uint32_t *launches);
// Wide builds (more than 2^lo_bits symbols in the collection): a text position is hi << lo_bits | lo with
// lo in the u32 value of the sort and hi (<= 8 bits) riding in the key bits from hi_shift upwards
// (hi_shift = 0: not wide); launch_heads then unloads hi into a byte array that travels with the suffix
// array through the refinement, like the BWT bytes do.

// Only the low key_bits of a key are compared.  If bwt != nullptr, bwt[i] = inv_map[code carried above
// the key bits] is written for every rank i.  diff (optional, head_words words): bit i = suffix i is not a
// group head and the carried symbol differs from that of suffix i-1, i.e. its group holds mixed BWT symbols.
void launch_heads(cudaStream_t st, int bits, const uint64_t *sorted_keys, uint64_t n, uint32_t *head,
                  uint64_t head_words, unsigned long long *remaining, int key_bits, const uint8_t *inv_map,
                  uint8_t *bwt, uint8_t *pos_hi, int hi_shift, uint32_t *diff, uint32_t *launches);

constexpr int kRefThreads = 256;
constexpr int kRefWindow = 1024;   // group heads owned by one CTA lie in a window of this many slots
constexpr int kRefGroupMaxWarps = 768; // larger groups go through the global path
// Slots of the head bitmap behind the last suffix (head_words_for), more than a window plus its largest
// group can reach; it also bounds a sort range: fewer than 2^32 - kRefCap - 64 suffixes.
constexpr int kRefCap = 2048;

inline uint64_t head_words_for(uint64_t n) { return div_up(n, 32) + kRefCap / 32 + 8; }

// One refinement round: every group of >= 2 suffixes that still agree on their
// first `depth` symbols is sorted (stably) by the next SPW symbols and split.
// head_next must hold a copy of head_cur.  Groups larger than kRefGroupMaxWarps are
// left untouched and their head slots appended to big_heads.  win_list (n_list
// entries; nullptr = every window) names the windows to visit; windows that
// still own unresolved groups afterwards are appended to win_next (deduplicated
// through the zeroed win_flag array, one u32 per window).  If bwt != nullptr the BWT bytes
// (one per rank) are permuted together with the suffix array.  A CTA keeps extending the keys
// (depth += SPW) until every group it owns is resolved, so that one launch finishes everything
// except the groups that do not fit a CTA.  full_order = false (default schedule, needs bwt): groups whose
// members all carry the same BWT symbol are left as they are -- their order cannot change the BWT -- so the
// suffix array is then only sorted as far as the BWT needs it.  diff_bits: launch_heads' bitmap while it is
// still valid (first launch after the initial sort), nullptr afterwards (the kernel then compares the bytes).
// big_groups: groups of 64+ members are ranked by the whole warp around their dominant key (kernels.cu, kRwBigGroup).
// Returns which instantiation of the kernel ran: kRwLaunched* bits and BITS << kRwLaunchedBitsShift (0: no window
// to visit, nothing launched).
constexpr uint32_t kRwLaunchedCoop = 2, kRwLaunchedWide = 4, kRwLaunchedOrder = 8, kRwLaunchedBitsShift = 8;
uint32_t launch_refine(cudaStream_t st, int bits, const uint64_t *packed, uint32_t *sa, const uint32_t *head_cur,
                   uint32_t *head_next, uint64_t n, uint32_t depth, const uint32_t *win_list, uint32_t n_list,
                   uint32_t *big_heads, uint32_t big_cap, uint32_t *big_count, unsigned long long *remaining,
                   uint32_t *win_flag, uint32_t *win_next, uint32_t *win_next_count, uint8_t *bwt, uint8_t *sa_hi,
                   int lo_bits, bool full_order, const uint32_t *diff_bits, uint32_t *launches, bool big_groups = false);

// BWT-only builds: the groups with mixed BWT symbols, copied out in order so that the refinement works on dense
// arrays.  launch_mark_active: act (zeroed, head_words words) gets the slots of those groups (diff is read 16 bytes
// at a time: aligned like every allocation of the builder), tile_off
// (active_tiles(words of n) + 1 entries) their running counts per tile, the total behind the last entry.
// launch_compact_active: fills the dense arrays (m_act entries; chi/sa_hi may be nullptr) and the compact
// head bitmap chead (zeroed by the caller, chead_words words, bits from m_act on set).
// launch_scatter_bwt: bwt[corig[j]] = cbw[j].
uint64_t active_tiles(uint64_t head_words);
void launch_mark_active(cudaStream_t st, const uint32_t *head, const uint32_t *diff, uint64_t n, uint32_t *act,
                        uint64_t *tile_off, uint32_t *launches);
void launch_compact_active(cudaStream_t st, const uint32_t *act, const uint32_t *head, uint64_t n, const uint64_t *tile_off,
                           const uint32_t *sa, const uint8_t *bwt, const uint8_t *sa_hi, uint64_t m_act, uint32_t *csa,
                           uint8_t *cbw, uint8_t *chi, uint32_t *corig, uint32_t *chead, uint64_t chead_words,
                           uint32_t *launches);
void launch_scatter_bwt(cudaStream_t st, const uint32_t *corig, const uint8_t *cbw, uint64_t m_act, uint8_t *bwt,
                        uint32_t *launches);

// Large-group path, step 1: length of each listed group (distance to the next head).
void launch_big_extent(cudaStream_t st, const uint32_t *head_cur, uint64_t n, const uint32_t *big_heads,
                       uint32_t nbig, uint32_t *big_len, uint32_t *launches);
// step 2: gather (suffix, next key, group ordinal) of all listed groups into dense arrays
void launch_big_gather(cudaStream_t st, int bits, const uint64_t *packed, const uint32_t *sa, uint32_t depth,
                       const uint32_t *big_heads, const uint64_t *big_off, uint32_t nbig, uint64_t total,
                       uint32_t *bsa, uint64_t *bkey, uint32_t *bgid, const uint8_t *sa_hi, uint8_t *bhi, int lo_bits,
                       uint32_t *launches);
// step 3 helper: k2[j] = gid[perm[j]]
void launch_gather_u32_to_u64(cudaStream_t st, const uint32_t *src, const uint32_t *perm, uint64_t n, uint64_t *dst,
                              uint32_t *launches);
// step 4: write the sorted groups back and mark the new heads
void launch_big_scatter(cudaStream_t st, int bits, const uint32_t *perm, const uint32_t *bsa, const uint64_t *bkey,
                        const uint32_t *bgid, const uint32_t *big_heads, const uint64_t *big_off, uint64_t total,
                        uint32_t *sa, uint32_t *head_next, uint32_t *win_flag, uint32_t *win_next,
                        uint32_t *win_next_count, const uint64_t *packed, const uint8_t *inv_map, uint8_t *bwt,
                        const uint8_t *bhi, uint8_t *sa_hi, int lo_bits, uint32_t *launches);

// out[i] = hi[i] << lo_bits | lo[i]  (hi may be nullptr)
void launch_widen_sa(cudaStream_t st, const uint32_t *lo, const uint8_t *hi, int lo_bits, uint64_t n, uint64_t *out,
                     uint32_t *launches);

// ---- BWT --------------------------------------------------------------------
// bwt[i] = byte of text[sa[i]-1], or 0 when suffix i is a whole document (incbwt/rlcsa.cpp:815-845);
// gathered from the packed text, inv_map[code] gives the byte back.
void launch_bwt(cudaStream_t st, int bits, const uint64_t *packed, const uint8_t *inv_map, const uint32_t *sa,
                uint64_t n, uint8_t *bwt, uint32_t *launches);

// ---- suffix-array samples (.sa; FMIndex::maketables, FMIndex.cpp:572-714) ---------------
// doc_end[k] = text position of document k's terminator; tile_scratch holds term_tiles(n) u64
uint64_t term_tiles(uint64_t n);
void launch_term_positions(cudaStream_t st, const uint8_t *raw, uint64_t n, uint64_t *tile_scratch, uint32_t *doc_end,
                           uint32_t *launches);
// mark (zeroed bitmap over text positions): sampled suffixes by the rule of FMIndex.cpp:624
void launch_sa_mark(cudaStream_t st, const uint32_t *doc_end, uint32_t ndocs, uint32_t rate, uint32_t *mark,
                    uint32_t *launches);
// out (u32 words, rank order): bit p = mark[sa[p]], or bwt[p] == 0 when mark is nullptr
void launch_sa_rank_bits(cudaStream_t st, const uint32_t *sa, const uint8_t *bwt, const uint32_t *mark, uint64_t n,
                         uint32_t *out, uint64_t out_words, uint32_t *launches);
// for every set bit p (j-th set bit): out_doc[j] = document of text position sa[p], out_off[j] = offset in it
void launch_sa_emit(cudaStream_t st, const uint32_t *sa, const uint64_t *bits, const uint64_t *Rs, const uint8_t *Rb,
                    uint64_t n, const uint32_t *doc_end, uint32_t ndocs, uint32_t *out_doc, uint32_t *out_off,
                    uint32_t *launches);

// The same tables for one slice of a packed-text build (slots of geom, launch_select).  Positions are u64 positions
// in the padded text; the first document of a slot starts at the slot's first symbol.
// doc_end[k] (u64) = padded position of document k's terminator, padding skipped; tile_scratch: term_tiles(n_text) u64
void launch_packed_term_positions(cudaStream_t st, int bits, const uint64_t *packed, uint64_t n_text, const SelGeom &geom,
                                  uint64_t *tile_scratch, uint64_t *doc_end, uint32_t *launches);
void launch_sa_mark64(cudaStream_t st, const uint64_t *doc_end, uint32_t ndocs, uint32_t rate, uint64_t slot_syms,
                      uint32_t *mark, uint32_t *launches);
// slice of m suffixes (position = hi << lo_bits | lo, hi may be nullptr): bit sampled_base + p of `sampled` (zeroed)
// = mark[position of p]; bit p of `ends` (zeroed) = bwt[p] == 0; counts[0] += set bits of sampled, counts[1] of ends
void launch_sa_slice_bits(cudaStream_t st, const uint32_t *sa, const uint8_t *hi, int lo_bits, const uint8_t *bwt,
                          const uint32_t *mark, uint64_t m, uint64_t *sampled, uint64_t sampled_base, uint64_t *ends,
                          unsigned long long *counts, uint32_t *launches);
// For every set bit q = bits_base + p (p < m) of `bits` with its directories: j = rank1(q) - rank_sub; the document
// k of the suffix's position is written as a doc_w-bit field at bit doc_bit0 + j * doc_w of doc_out (zeroed), its
// offset in k (when off_out) as an off_w-bit field at off_bit0 + j * off_w of off_out.
void launch_sa_emit64(cudaStream_t st, const uint32_t *sa, const uint8_t *hi, int lo_bits, const uint64_t *bits,
                      const uint64_t *Rs, const uint8_t *Rb, uint64_t bits_base, uint64_t rank_sub, uint64_t m,
                      const uint64_t *doc_end, uint32_t ndocs, uint64_t slot_syms, uint64_t *doc_out, uint64_t doc_bit0,
                      unsigned doc_w, uint64_t *off_out, uint64_t off_bit0, unsigned off_w, uint32_t *launches);
// lengths (terminator excluded) of documents [first, first + count) as w-bit fields from bit bit0 of out (zeroed)
void launch_sa_lengths(cudaStream_t st, const uint64_t *doc_end, uint64_t first, uint64_t count, uint64_t slot_syms,
                       uint64_t *out, uint64_t bit0, unsigned w, uint32_t *launches);

// ---- wavelet tree -------------------------------------------------------------
constexpr int kWtTile = 8192; // symbols per CTA
constexpr int kWtMaxNodes = 255;

// node_info[v*256 + c]: 0 = symbol c not below internal node v, 1 = member with bit 0, 3 = member with bit 1
void launch_wt_count(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                     uint64_t ntiles, uint64_t *tile_count, uint32_t *launches);
// in-place exclusive scan of tile_count[v][0..ntiles) for every node v
void launch_wt_scan(cudaStream_t st, uint64_t *tile_count, int n_internal, uint64_t ntiles, uint32_t *launches);
// node_data[v] = device pointer of node v's (zeroed) bit array; node_ch[v] receives the first member symbol
// bit_base[v] (optional, device): bit offset of the sequence's first member inside node_data[v] (multi-GPU pieces)
void launch_wt_fill(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                    uint64_t ntiles, const uint64_t *tile_off, uint64_t *const *node_data, uint8_t *node_ch,
                    const uint64_t *bit_base, uint32_t *launches);

// Trees of at most 8 internal nodes: count, scan and fill in ONE pass over the sequence (decoupled look-back over
// the tiles, the tile's bits assembled in shared memory).  status: wt_sweep_status_words(ntiles) u64, counter: one u32.
bool wt_sweep_ok(int n_internal);
uint64_t wt_sweep_status_words(uint64_t ntiles);
void launch_wt_sweep(cudaStream_t st, const uint8_t *seq, uint64_t n, const uint8_t *node_info, int n_internal,
                     uint64_t ntiles, uint64_t *status, uint32_t *counter, uint64_t *const *node_data, uint8_t *node_ch,
                     const uint64_t *bit_base, uint32_t *launches);

// Multi-GPU: node bit arrays arrive as pieces built on different GPUs.  nwords words from src + src_word
// are merged into dst (first / last word OR-ed, interior copied); gridDim.y = pieces.
struct WtPiece {
    uint64_t src_word;
    uint64_t *dst;
    uint64_t nwords;
};
void launch_wt_merge_pieces(cudaStream_t st, const uint64_t *src, const WtPiece *pieces, uint32_t npieces,
                            uint32_t *launches);

// BitRank directories of one bit array (BitRank.cpp:154-187): Rs[j] = ones in
// words [0,4j), j <= nbits/256; Rb[k] = ones in words [4*(k/4), k), k <= nbits/64.
// `scratch` holds ceil((nbits/256+1)/kRankChunk)+1 u64.
constexpr int kRankChunk = 2048; // superblocks per CTA
// `base` is added to every Rs entry (ones in front of the array when it is a piece of a longer bit vector).
void launch_bitrank(cudaStream_t st, const uint64_t *data, uint64_t nbits, uint64_t *Rs, uint8_t *Rb,
                    uint64_t *scratch, uint32_t *launches, uint64_t base = 0);

} // namespace dsmfm
