/*
 * dsmfm.h -- C ABI of the B200-native FM-index construction path.
 *
 * This is the drop-in boundary for ONE path of HIITMetagenomics/dsm-framework:
 * what `builder -v input.fasta` does between TextCollectionBuilder::InsertText
 * and the bytes of the `.fmi` file.  The reference has no plugin ABI for this
 * path -- it is a C++ class (TextCollectionBuilder.h:41-73) over incbwt -- so
 * the entry points below are what a binding from the reference's C++ facade
 * binds; INTEGRATION.md shows that binding.  Each entry point cites the
 * reference interface it replaces (file:line relative to the reference tree).
 *
 * Plain C, plain pointers and sizes; no CUDA, torch or C++ types.  All entry
 * points return 0 on success or a negative DSMFM_E* code; the message is then
 * available from dsmfm_last_error().  There is NO CPU fallback: without a
 * usable sm_100 device dsmfm_create fails with DSMFM_ECUDA.
 *
 * Threading: one builder per thread, not re-entrant per handle (the reference
 * is "not thread-safe" as well, builder.cpp:266).
 */
#ifndef DSMFM_H_
#define DSMFM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSMFM_API __attribute__((visibility("default")))

#define DSMFM_VERSION 1

enum {
    DSMFM_OK = 0,
    DSMFM_EINVAL = -1,  /* bad argument / call order (e.g. append after finish) */
    DSMFM_ECUDA = -2,   /* CUDA runtime error, or no usable device            */
    DSMFM_ENOMEM = -3,  /* host or device allocation failed                    */
    DSMFM_EEMPTY = -4,  /* an empty document was inserted                      */
    DSMFM_ELIMIT = -5,  /* input exceeds a limit of this build (see message)   */
    DSMFM_EIO = -6      /* file write error                                    */
};

/* Default SA sample rate written into the .fmi header
 * (TEXTCOLLECTION_DEFAULT_SAMPLERATE, TextCollectionBuilder.h:30). */
#define DSMFM_DEFAULT_SAMPLERATE 124

typedef struct dsmfm_builder dsmfm_builder;

typedef struct dsmfm_options {
    int32_t device;          /* CUDA device ordinal; -1 = current device                         */
    uint32_t samplerate;     /* 0 -> 124, as TextCollectionBuilder.cpp:37-39                      */
    uint64_t expected_bytes; /* hint: total bytes of documents incl. terminators (0 = unknown)    */
    void *stream;            /* cudaStream_t to run on; NULL = the builder creates a non-blocking  */
                             /* stream of its own (NULL + DSMFM_FLAG_DEFAULT_STREAM: the legacy    */
                             /* default stream).  Everything the builder does is ordered on this   */
                             /* stream ONLY: device buffers handed to dsmfm_append_batch_device /   */
                             /* dsmfm_build_packed must be complete on it, i.e. produced on it or   */
                             /* synchronised with it by the caller before the call                  */
    uint32_t flags;          /* DSMFM_FLAG_*                                                      */
    uint32_t reserved;
    /* Key-range sharding of ONE collection over several GPUs (one builder per GPU, every builder is
     * given the WHOLE collection): the suffixes are cut into `shard_count` ranges of their first key
     * with about equal population; this builder sorts ranges [shard_index, shard_index + shard_span)
     * one after the other and produces the matching contiguous slice of the global suffix array / BWT
     * (dsmfm_shard_info).  shard_count 0 or 1 = the whole index on this GPU (limit: 2^32 symbols).
     * Sharded builds index collections of up to 2^40 symbols; each single range must hold fewer than
     * 2^32 suffixes and bounds the sort buffers (24 bytes x 2 per suffix of the range), so G GPUs
     * with K ranges each use shard_count = G*K, shard_index = g*K, shard_span = K. */
    uint32_t shard_index;
    uint32_t shard_count;
    uint32_t shard_span;     /* 0 -> 1 */
    uint32_t reserved2;
} dsmfm_options;

#define DSMFM_FLAG_KEEP_BWT 1u /* keep the plain BWT in host memory after finish (dsmfm_index.bwt)   */
#define DSMFM_FLAG_KEEP_SA 2u  /* keep suffix array, BWT and document boundaries on the device (dsmfm_write_sa, dsmfm_sa_*) */
#define DSMFM_FLAG_DEFAULT_STREAM 4u /* opts->stream == NULL names the legacy default stream, not "create one" */

/* One Huffman code-table entry: HuffWT::TCodeEntry, HuffWT.h:13-19. */
typedef struct dsmfm_code {
    uint64_t count;
    uint32_t bits;
    uint32_t code;
} dsmfm_code;

/* One wavelet-tree node in pre-order: HuffWT members (HuffWT.h:48-53) plus its
 * BitRank (BitRank.h:19-24).  For a leaf only `leaf` and `ch` are meaningful. */
typedef struct dsmfm_node {
    uint8_t leaf;
    uint8_t ch;            /* first symbol of the node's subsequence (HuffWT.cpp:8) */
    uint8_t pad[6];
    uint64_t nbits;        /* BitRank::n                                             */
    uint64_t integers;     /* BitRank::integers = ceil((n+1)/64)                     */
    const uint64_t *data;  /* [integers]                                             */
    const uint64_t *Rs;    /* [nbits/256 + 1]                                        */
    const uint8_t *Rb;     /* [nbits/64 + 1]                                         */
} dsmfm_node;

/* Everything FMIndex::save (FMIndex.cpp:155-217) writes, as host pointers that
 * stay valid until dsmfm_destroy. */
typedef struct dsmfm_index {
    uint64_t n;              /* indexed symbols incl. terminators (FMIndex::n)           */
    uint32_t samplerate;
    uint32_t number_of_texts;
    uint64_t max_text_length;
    uint64_t C[256];         /* FMIndex.cpp:397-409                                      */
    dsmfm_code codetable[256];
    uint32_t n_nodes;
    uint32_t reserved;
    const dsmfm_node *nodes; /* pre-order, n_nodes entries                               */
    const uint8_t *bwt;      /* [n] if DSMFM_FLAG_KEEP_BWT, else NULL                    */
} dsmfm_index;

/* Per-build measurements (device times from CUDA events on the build stream). */
typedef struct dsmfm_stats {
    uint64_t n;                  /* indexed symbols                                        */
    uint64_t bases;              /* sum of document lengths excl. terminators              */
    uint32_t bits_per_symbol;    /* 3, 4 or 8                                               */
    uint32_t sigma;              /* distinct non-terminator symbols                        */
    uint32_t rounds;             /* refinement rounds run after the initial sort           */
    uint32_t kernel_launches;    /* kernels launched by the build (our own kernels only)   */
    uint64_t active[32];         /* suffixes in non-singleton groups entering round r      */
    uint64_t fallback_elems;     /* suffixes that went through the large-group path        */
    float ms_total;              /* whole device build                                      */
    float ms_pack;               /* histogram + pack                                        */
    float ms_sort;               /* key build + LSD radix sort + head marking               */
    float ms_sort_pass;          /* mean duration of one onesweep LAUNCH (dominant kernel)  */
    float ms_refine;             /* all refinement rounds                                   */
    float ms_bwt;                /* BWT emission                                            */
    float ms_wt;                 /* wavelet tree + BitRank directories                      */
    float ms_h2d;                /* last finish: host->device copies not overlapped         */
    float ms_d2h;                /* last finish: device->host of the sections               */
    uint32_t sort_passes;        /* LSD passes of the initial sort (of the last key range)  */
    uint32_t sort_launches;      /* onesweep launches of the initial sorts: a pass over more */
                                 /* than 2^29 pairs runs as several launches                 */
    uint64_t sort_pass_bytes;    /* mean algorithmic bytes moved by ONE onesweep launch      */
    uint64_t device_bytes_peak;  /* peak device memory held by the builder                  */
    float ms_wall_build;         /* host wall time of dsmfm_build_device                    */
    float ms_wall_fetch;         /* host wall time of dsmfm_fetch                           */
    float ms_wall_alloc;         /* of which: device allocation calls                       */
    uint32_t streamed;           /* 1: the text streamed in from the host in pieces and was packed and keyed   */
                                 /* piece by piece behind the copy (dsmfm_append_batch of a whole collection)  */
    uint64_t refine_key_fetches; /* 8-byte keys the refinement kernel gathered from the text */
    uint64_t refine_launches;    /* refine_kernel launches                                  */
    uint64_t refine_members;     /* suffixes in the tie groups that had to be sorted: all of them when the */
                                 /* suffix array is kept, else those of groups with mixed BWT symbols       */
} dsmfm_stats;

/* Replaces: TextCollectionBuilder::TextCollectionBuilder (TextCollectionBuilder.cpp:32-57). */
DSMFM_API int dsmfm_create(const dsmfm_options *opts, dsmfm_builder **out);

/* Replaces: TextCollectionBuilder::InsertText -> RLCSABuilder::insertSequence
 * (TextCollectionBuilder.cpp:65-98; incbwt/rlcsa_builder.cpp:36-78).
 * `doc` holds `len` symbols from [1,255] (no terminator); it is copied.  The
 * i-th call gets document id i-1.  len == 0 -> DSMFM_EEMPTY (the reference
 * prints an error and exits, TextCollectionBuilder.cpp:86-91). */
DSMFM_API int dsmfm_append(dsmfm_builder *b, const uint8_t *doc, size_t len);

/* Bulk form of dsmfm_append: `bytes` bytes holding documents each followed by
 * one '\0' (the layout RLCSABuilder keeps in its buffer, rlcsa_builder.cpp:54-60).
 * The last byte must be '\0'.  Document count and longest length are taken on
 * the device.  The host-to-device copy is asynchronous when `docs` is page-locked: the buffer must stay
 * unchanged until the build has synchronised (dsmfm_build_device / dsmfm_finish return). */
DSMFM_API int dsmfm_append_batch(dsmfm_builder *b, const uint8_t *docs, size_t bytes);

/* Same, but `docs` is DEVICE memory on the builder's device (inputs already
 * resident in HBM); copied device-to-device on the builder's stream.  The copy is ordered after earlier
 * work of THAT stream only: a buffer filled on another stream (a collective, another library) must be
 * complete -- synchronise, or make the builder's stream wait on an event -- before this call.  The buffer
 * may be released once the builder's stream has consumed the copy (dsmfm_build_device synchronises it). */
DSMFM_API int dsmfm_append_batch_device(dsmfm_builder *b, const void *docs_dev, size_t bytes);

/* Replaces: the record loop and per-read transform of the reference CLI, build() in builder.cpp:203-262
 * with normalize() (60-104) and transform() (183-201) -- SURVEY 8(f) row 3, the step in front of InsertText.
 * `text` holds `len` bytes of a FASTA file (host memory).  On the device, every record with a non-empty
 * sequence s becomes the document complement(s) + '-' + reverse(s) + '\0' and is appended to the
 * collection in file order, exactly the bytes the reference's loop hands to InsertText: rows are split
 * at '\n' only ('\r' stays in the sequence and is normalised to N like any other foreign symbol), rows
 * in front of the first header form a record of their own, records without sequence are skipped.
 * final != 0: everything is parsed; a last row without '\n' is dropped, as `getline(...).good()` drops it
 * (builder.cpp:211).  final == 0 (streaming): only the bytes in front of the last header line are parsed,
 * info->consumed says how many; present the rest again, followed by more input. */
typedef struct dsmfm_fasta_info {
    uint64_t consumed;             /* bytes of `text` this call has dealt with                            */
    uint64_t records;              /* header lines seen                                                   */
    uint64_t documents;            /* documents appended (records with a non-empty sequence)              */
    uint64_t bases;                /* sequence symbols                                                    */
    uint64_t doc_bytes;            /* bytes appended to the collection (documents incl. terminators)      */
    uint64_t invalid_records;      /* records holding symbols outside ACGTNacgtn0123. (they become N)      */
    uint64_t first_invalid_offset; /* offset in `text` of the first such symbol, ~0 if none               */
    uint64_t bad_headers;          /* header lines with nothing but blanks after '>': the reference throws */
                                   /* std::out_of_range on them (builder.cpp:215)                          */
} dsmfm_fasta_info;
DSMFM_API int dsmfm_append_fasta(dsmfm_builder *b, const uint8_t *text, size_t len, int final, dsmfm_fasta_info *info);

/* Replaces: TextCollectionBuilder::InitTextCollection -> RLCSABuilder::getBWT
 * -> FMIndex::FMIndex -> makewavelet -> HuffWT::makeHuffWT -> BitRank::BuildRank
 * (TextCollectionBuilder.cpp:100-152; rlcsa_builder.cpp:166-179; FMIndex.cpp:92-123,
 * 395-425; HuffWT.cpp:5-55,133-192; BitRank.cpp:89-103,154-187).
 * Runs the whole device path and returns the finished sections in host
 * memory.  No documents -> the reference's one-symbol "\0" index
 * (TextCollectionBuilder.cpp:111-119).  Further appends fail. */
DSMFM_API int dsmfm_finish(dsmfm_builder *b, dsmfm_index *out);

/* The two halves of dsmfm_finish, for measuring the device path alone:
 * dsmfm_build_device runs every kernel and leaves the sections in HBM;
 * dsmfm_fetch copies them to the host and fills `out`. */
DSMFM_API int dsmfm_build_device(dsmfm_builder *b);
DSMFM_API int dsmfm_fetch(dsmfm_builder *b, dsmfm_index *out);

/* ---- one collection over several GPUs (no counterpart in the single-process reference) ----
 * After dsmfm_build_device on a sharded builder: the slice of the global suffix order it owns. */
typedef struct dsmfm_shard {
    uint64_t n_total;     /* symbols of the whole collection                                  */
    uint64_t rank_begin;  /* global rank of the first suffix of this slice                    */
    uint64_t count;       /* suffixes in this slice                                           */
    const void *bwt_dev;  /* DEVICE pointer: BWT bytes of the slice [count]                   */
    const void *sa_dev;   /* reserved (use dsmfm_shard_export for the suffix array)           */
} dsmfm_shard;
DSMFM_API int dsmfm_shard_info(dsmfm_builder *b, dsmfm_shard *out);

/* Copies the slice into caller-provided DEVICE buffers on the builder's device (either may be NULL),
 * on the builder's stream, and waits for the copy: bwt_dst_dev[count] bytes; sa_dst_dev[count]
 * text positions as u64 (needs DSMFM_FLAG_KEEP_SA). */
DSMFM_API int dsmfm_shard_export(dsmfm_builder *b, void *bwt_dst_dev, void *sa_dst_dev);

/* On the assembling GPU: build C[], the code table, the wavelet tree and the BitRank directories
 * from the concatenated BWT (`bwt_dev`, device memory, n_total bytes, slices in shard order).
 * dsmfm_fetch then returns the index of the whole collection. */
DSMFM_API int dsmfm_assemble(dsmfm_builder *b, const void *bwt_dev, uint64_t n_total);

/* ---- wavelet tree built by several GPUs ----
 * Instead of shipping whole BWT slices to one GPU (dsmfm_assemble), every GPU turns its slice into
 * the bits it contributes to each wavelet-tree node ("pieces", about 0.28 bytes per symbol), already
 * shifted to their global bit offset modulo 64; the assembling GPU copies them into place and builds
 * the BitRank directories.  All that has to be agreed on is the table hist_all[world][256] of the
 * slices' byte histograms (dsmfm_slice_hist of every builder, in slice order).
 *   dsmfm_pieces_bytes(b, hist_all, world, r)      size of builder r's piece buffer (r == world: sum of all)
 *   dsmfm_build_pieces(b, hist_all, world, r, dst) fills dst (DEVICE memory of that size) on builder r
 *   dsmfm_assemble_pieces(b, hist_all, world, src) src = the world piece buffers back to back in slice
 *                                                  order (DEVICE memory); dsmfm_fetch then returns the index */
DSMFM_API int dsmfm_slice_hist(dsmfm_builder *b, uint64_t *out256);
DSMFM_API uint64_t dsmfm_pieces_bytes(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank);
DSMFM_API int dsmfm_build_pieces(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank, void *dst_dev);
DSMFM_API int dsmfm_assemble_pieces(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, const void *pieces_dev);

/* ---- one collection over several GPUs, packed-text exchange (what bench.py --gpus N and `builder --gpus N` run) ----
 * Replaces, across GPUs, incbwt's batch merge -- RLCSABuilder::addRLCSA / getRanks / mergeRLCSA
 * (incbwt/rlcsa_builder.cpp:245-318; incbwt/rlcsa.cpp:156-220, 307-337) -- whose result is, like everything on this
 * path, a function of the text alone: builder r of `world` holds block r of the documents (block order = document
 * order).  Nothing but small tables and the PACKED blocks (3 bits per symbol for reads) has to travel:
 *   1. dsmfm_block_stats      every builder: histogram / document count / longest document of its block
 *      -> all-gather the dsmfm_block_info records (any transport: NCCL, MPI, shared memory of a threaded host)
 *   2. dsmfm_text_plan        pure host arithmetic, identical on every builder: alphabet, bits per symbol, the slot
 *                             every block occupies in the packed text (equal slots, so one all-gather moves them)
 *   3. dsmfm_block_pack       every builder packs ITS block into its slot of `text_dev` (device buffer holding the
 *                             whole packed text) and counts the top 12 key bits of its suffixes (4096 bins)
 *      -> all-gather the slots (in place), sum the 4096-bin histograms over the builders
 *   4. dsmfm_build_packed     every builder sorts the key ranges dsmfm_options.shard_* name, reading the replicated
 *                             packed text; dsmfm_shard_info / dsmfm_slice_hist describe its slice of the global BWT
 *      -> all-gather the slice histograms
 *   5. dsmfm_pieces_build     every builder: its slice's share of every wavelet-tree node -- bit words, Rs, Rb with
 *                             the counts of the slices in front of it added -- built on ITS GPU and copied to ITS host
 *      -> all-gather the dsmfm_piece_edge records (12 words per node and builder)
 *   6. dsmfm_pieces_merge     host: words and directory entries next to a slice boundary are completed
 *   7. dsmfm_pieces_write     every builder writes its share straight into `<prefix>.fmi` (pwrite at the offsets of
 *                             FMIndex::save's layout, FMIndex.cpp:155-217); the builder given `header` != 0 adds the rest.
 *   8-11. (DSMFM_FLAG_KEEP_SA) the same for the `.sa` samples: dsmfm_sa_slice_info, dsmfm_sa_pieces_build /
 *                             _merge / _write, below.
 * No builder ever holds the whole index, no GPU the whole wavelet tree, and the device-to-host copies run in parallel. */
#define DSMFM_MAX_BLOCKS 64

typedef struct dsmfm_block_info {
    uint64_t counts[256];       /* byte histogram of the block                                       */
    uint64_t bytes;             /* symbols incl. terminators                                         */
    uint64_t documents;
    uint64_t max_text_length;   /* longest document incl. its terminator                             */
    uint32_t empty_document;    /* the block holds an empty document (two terminators in a row)      */
    uint32_t reserved;
} dsmfm_block_info;

typedef struct dsmfm_text_plan {
    uint32_t world;
    uint32_t bits;              /* bits per packed symbol: 3, 4 or 8                                 */
    uint64_t n;                 /* symbols of the collection                                         */
    uint64_t documents;
    uint64_t max_text_length;
    uint64_t slot_words;        /* 64-bit words per slot (the same for every block)                  */
    uint64_t text_bytes;        /* size of the packed-text buffer: (world * slot_words + 8) * 8      */
    uint64_t counts[256];       /* histogram of the collection                                       */
    uint64_t block_bytes[DSMFM_MAX_BLOCKS];
} dsmfm_text_plan;

/* Further appends fail.  Synchronises the builder's stream. */
DSMFM_API int dsmfm_block_stats(dsmfm_builder *b, dsmfm_block_info *out);
/* DSMFM_EEMPTY if any block holds an empty document, DSMFM_EINVAL if world is 0 or above DSMFM_MAX_BLOCKS. */
DSMFM_API int dsmfm_text_plan_make(const dsmfm_block_info *all, uint32_t world, dsmfm_text_plan *out);
/* text_dev: DEVICE memory of plan->text_bytes on the builder's device; words [rank*slot_words, (rank+1)*slot_words)
 * are written (the block, then zeros).  top_hist4096: HOST array, the block's counts are stored (not added).
 * The builder's raw block is released.  Synchronises the builder's stream. */
DSMFM_API int dsmfm_block_pack(dsmfm_builder *b, const dsmfm_text_plan *plan, uint32_t rank, void *text_dev,
                               uint64_t *top_hist4096);
/* text_dev must be complete on the builder's stream (all slots, and 8 zero words behind the last slot) and stay
 * untouched until the call returns; top_hist4096 = the sum over all builders.  With DSMFM_FLAG_KEEP_SA the slice is
 * sorted in full order and what the .sa samples need is derived before the call returns (dsmfm_sa_*, step 8 on). */
DSMFM_API int dsmfm_build_packed(dsmfm_builder *b, const dsmfm_text_plan *plan, const void *text_dev,
                                 const uint64_t *top_hist4096);

typedef struct dsmfm_piece_edge {   /* one per internal node of the wavelet tree and builder; all-gathered */
    uint64_t count;                 /* members of the node in this builder's slice (0: the rest is void)   */
    uint64_t first_word;            /* first data word the slice contributes bits to                       */
    uint64_t first[4];              /* its contribution to words first_word .. first_word + 3              */
    uint64_t last_word;             /* last data word it contributes bits to                               */
    uint64_t last[4];               /* its contribution to words last_word - 3 .. last_word                */
    uint64_t ch;                    /* first member symbol of the slice (HuffWT.cpp:8)                     */
} dsmfm_piece_edge;

typedef struct dsmfm_piece {        /* this builder's share of one internal node's BitRank (BitRank.h:19-24) */
    uint32_t node;                  /* index in the pre-order node list of the index                        */
    uint32_t reserved;
    uint64_t word_first, word_count; /* data[word_first .. word_first + word_count)                          */
    uint64_t rs_first, rs_count;     /* Rs[rs_first .. )                                                     */
    uint64_t rb_first, rb_count;     /* Rb[rb_first .. )                                                     */
    uint64_t *data;                  /* HOST memory, valid until dsmfm_destroy; final after dsmfm_pieces_merge */
    uint64_t *Rs;
    uint8_t *Rb;
} dsmfm_piece;

typedef struct dsmfm_pieces {
    uint32_t n_internal;            /* internal nodes of the tree = entries of `piece` and `edge`           */
    uint32_t world, rank;
    uint32_t reserved;
    uint64_t bytes;                 /* bytes of sections this builder holds (copied device to host)         */
    const dsmfm_piece *piece;
    const dsmfm_piece_edge *edge;   /* this builder's records for the exchange                              */
} dsmfm_pieces;

/* hist_all[world][256]: dsmfm_slice_hist of every builder, in slice order.  The device work; with out != NULL the
 * sections are copied to the host right away (dsmfm_pieces_fetch), with out == NULL they stay in HBM until then. */
DSMFM_API int dsmfm_pieces_build(dsmfm_builder *b, const uint64_t *hist_all, uint32_t world, uint32_t rank, dsmfm_pieces *out);
DSMFM_API int dsmfm_pieces_fetch(dsmfm_builder *b, dsmfm_pieces *out);
/* edges_all[world][n_internal] in slice order (host). */
DSMFM_API int dsmfm_pieces_merge(dsmfm_builder *b, const dsmfm_piece_edge *edges_all, uint32_t world);
/* The header fields, C[], code table and node list (leaf / ch / nbits / integers; data pointers NULL) of the whole
 * index, as every builder knows them after dsmfm_pieces_merge. */
DSMFM_API int dsmfm_pieces_index(dsmfm_builder *b, dsmfm_index *out);
/* Writes this builder's share into `<path_prefix>.fmi` (created if missing, never truncated: every builder of the
 * build writes the same file, in any order).  header != 0: also everything that is not a BitRank array, and the
 * file is cut to its final size. */
DSMFM_API int dsmfm_pieces_write(dsmfm_builder *b, const char *path_prefix, int header);

/* ---- the .sa samples of a packed-text build (builders created with DSMFM_FLAG_KEEP_SA) ----
 * The `.sa` file (dsmfm_write_sa) is five bit vectors: `sampled` (a BitRank over the n BWT positions), then the
 * BlockArrays `suffixes` and `suffixDocId` (one field per sample, in BWT order), `textLength` (per document) and `Doc`
 * (per end marker, in BWT order).  Every builder holds a contiguous range of each: its BWT slice of `sampled`, the
 * fields of its slice's samples and end markers, the lengths of its block's documents.  dsmfm_build_packed derives
 * what needs the text or the BWT (document ends of the whole collection, the slice's sampled and end-marker bits);
 * after the .fmi steps (or instead of them):
 *   8. dsmfm_sa_slice_info    every builder: samples / end markers of its slice, documents of its block
 *      -> all-gather the dsmfm_sa_info records
 *   9. dsmfm_sa_pieces_build  every builder: its share of the five vectors at their global bit offsets (the Rs of
 *                             `sampled` with the samples of earlier slices added), copied to its host; returns one
 *                             dsmfm_piece_edge per vector
 *      -> all-gather the edge records (DSMFM_SA_VECTORS per builder)
 *  10. dsmfm_sa_pieces_merge  host: words and directory entries next to a slice boundary are completed
 *  11. dsmfm_sa_pieces_write  every builder writes its share into `<prefix>.sa` (pwrite, never truncates); the builder
 *                             given `header` != 0 adds the file header and the four BlockArray headers and cuts the
 *                             file to its size.
 * Document ids are u32 in the file's readers: collections of 2^32 documents or more are refused (DSMFM_ELIMIT). */
#define DSMFM_SA_VECTORS 5

typedef struct dsmfm_sa_info {
    uint64_t samples;   /* sampled suffixes in this builder's BWT slice          */
    uint64_t ends;      /* end markers (BWT symbol 0) in the slice               */
    uint64_t documents; /* documents of this builder's block                     */
} dsmfm_sa_info;

DSMFM_API int dsmfm_sa_slice_info(dsmfm_builder *b, dsmfm_sa_info *out);
/* infos_all[world]: dsmfm_sa_slice_info of every builder, in slice order.  edges_out[DSMFM_SA_VECTORS]. */
DSMFM_API int dsmfm_sa_pieces_build(dsmfm_builder *b, const dsmfm_sa_info *infos_all, uint32_t world, uint32_t rank,
                                    dsmfm_piece_edge *edges_out);
/* edges_all[world][DSMFM_SA_VECTORS] in slice order (host). */
DSMFM_API int dsmfm_sa_pieces_merge(dsmfm_builder *b, const dsmfm_piece_edge *edges_all, uint32_t world);
DSMFM_API int dsmfm_sa_pieces_write(dsmfm_builder *b, const char *path_prefix, int header);

/* Helpers for hosts that do not link the CUDA runtime themselves (the C++ CLI runs one thread per GPU and moves
 * the packed slots with peer copies instead of NCCL): device memory for the packed text, and the copy of slot
 * `rank` of this builder's text into the text buffer of another device (peer-to-peer over NVLink when the devices
 * allow it), ordered on the builder's stream and waited for. */
DSMFM_API int dsmfm_device_count(void);
DSMFM_API void *dsmfm_device_alloc(int device, size_t bytes);
DSMFM_API void dsmfm_device_free(int device, void *p);
DSMFM_API int dsmfm_slot_send(dsmfm_builder *b, const dsmfm_text_plan *plan, uint32_t rank, const void *text_src_dev,
                              int dst_device, void *text_dst_dev);

/* Replaces: FMIndex::save (FMIndex.cpp:155-217).  Writes `<path_prefix>.fmi`
 * byte-for-byte in the reference layout (version 17). */
DSMFM_API int dsmfm_write_fmi(const dsmfm_index *idx, const char *path_prefix);

/* Replaces: FMIndex::saveSamples -> FMIndex::maketables (FMIndex.cpp:125-147, 572-714), the SA sampling
 * the reference builder leaves dormant.  Writes `<path_prefix>.sa`: BitRank `sampled` (one bit per BWT
 * position), BlockArray `suffixes` (offset of each sampled suffix in its document), `suffixDocId`,
 * `textLength`, and `Doc` (document of every end marker in BWT order), byte for byte what the reference
 * writes at the index's sample rate.  Needs DSMFM_FLAG_KEEP_SA on an unsharded builder, after
 * dsmfm_finish; the tables are derived on the device from the suffix array. */
DSMFM_API int dsmfm_write_sa(dsmfm_builder *b, const char *path_prefix);
DSMFM_API uint64_t dsmfm_sa_size(dsmfm_builder *b);
DSMFM_API int dsmfm_sa_serialize(dsmfm_builder *b, uint8_t *out, uint64_t out_cap);

/* Serialise the same bytes into memory.  dsmfm_fmi_size gives the exact size. */
DSMFM_API uint64_t dsmfm_fmi_size(const dsmfm_index *idx);
DSMFM_API int dsmfm_fmi_serialize(const dsmfm_index *idx, uint8_t *out, uint64_t out_cap);

/* Copy suffix-array entries [first, first+count) (text positions) to the host;
 * needs DSMFM_FLAG_KEEP_SA.  For tests and the .sa writer. */
DSMFM_API int dsmfm_copy_sa(dsmfm_builder *b, uint32_t *out, uint64_t first, uint64_t count);

DSMFM_API int dsmfm_get_stats(const dsmfm_builder *b, dsmfm_stats *out);

/* Message of the last failure on this handle (or of a failed dsmfm_create when b == NULL). */
DSMFM_API const char *dsmfm_last_error(const dsmfm_builder *b);

/* Replaces: TextCollectionBuilder::~TextCollectionBuilder + ~FMIndex. */
DSMFM_API void dsmfm_destroy(dsmfm_builder *b);

DSMFM_API int dsmfm_version(void);

/* Device and pinned host memory are cached between builds (a second build of the
 * same size allocates nothing).  This returns the cached memory of `device`
 * (-1 = all devices) to the system. */
DSMFM_API int dsmfm_release_cached(int device);

/* ---- the query half of the index on the GPU (SURVEY 8f row 1) -------------------------------------------
 * Replaces, for batches of queries, what the mining client (metaenumerate, EnumerateQuery.cpp:39-58, 105-149;
 * Query.h:37-45) asks of a loaded index: FMIndex::LF and getL (FMIndex.h:84-102) over HuffWT::rank / access
 * (HuffWT.h:66-83, 125-157) and BitRank::rank (BitRank.cpp:191-195).  The wavelet tree stays in HBM in the
 * layout of the .fmi file.  All arrays are HOST memory of `count` entries unless stated otherwise; positions
 * wrap like the reference's unsigned longs (rank / LF at i = (uint64_t)-1 count nothing). */
typedef struct dsmfm_searcher dsmfm_searcher;
/* from the sections dsmfm_finish / dsmfm_fetch returned (uploads them) */
DSMFM_API int dsmfm_searcher_create(int device, const dsmfm_index *idx, dsmfm_searcher **out);
/* Replaces: TextCollection::load -> FMIndex::FMIndex(FILE *) (TextCollection.cpp:27-62; FMIndex.cpp:245-357;
 * HuffWT.cpp:57-71, 201-207; BitRank.cpp:111-132) for what the queries need: n, C, code table, tree. */
DSMFM_API int dsmfm_searcher_open(int device, const char *fmi_path, dsmfm_searcher **out);
DSMFM_API uint64_t dsmfm_searcher_length(const dsmfm_searcher *s);
/* out[k] = HuffWT::rank(c[k], i[k]): occurrences of c[k] in BWT[0 .. i[k]] */
DSMFM_API int dsmfm_searcher_rank(dsmfm_searcher *s, const uint8_t *c, const uint64_t *i, uint64_t *out, uint64_t count);
/* out[k] = FMIndex::LF(c[k], i[k]) = C[c] + rank_c(i) */
DSMFM_API int dsmfm_searcher_lf(dsmfm_searcher *s, const uint8_t *c, const uint64_t *i, uint64_t *out, uint64_t count);
/* the same with DEVICE arrays on the searcher's device (no copies; for measuring the kernel) */
DSMFM_API int dsmfm_searcher_lf_device(dsmfm_searcher *s, const void *c_dev, const void *i_dev, void *out_dev, uint64_t count);
/* sym[k] = FMIndex::getL(i[k]); rank[k] (may be NULL) = its rank, as HuffWT::access(i, rank) returns it */
DSMFM_API int dsmfm_searcher_access(dsmfm_searcher *s, const uint64_t *i, uint8_t *sym, uint64_t *rank, uint64_t count);
/* Query::pushChar for every symbol of `symbols` at once: interval k extended to the left by symbols[j] is
 * [sp_out, ep_out][k * nsym + j] = [LF(c, sp-1), LF(c, ep)-1]; empty intervals (sp > ep) pass through. */
DSMFM_API int dsmfm_searcher_extend(dsmfm_searcher *s, const uint64_t *sp, const uint64_t *ep, uint64_t count,
                                    const uint8_t *symbols, uint32_t nsym, uint64_t *sp_out, uint64_t *ep_out);
/* backward search of whole patterns (pattern k = patterns[offsets[k] .. offsets[k+1])), last symbol first, from
 * the interval of all suffixes: [sp, ep] of its occurrences, sp > ep if there are none */
DSMFM_API int dsmfm_searcher_count(dsmfm_searcher *s, const uint8_t *patterns, const uint64_t *offsets, uint64_t count,
                                   uint64_t *sp_out, uint64_t *ep_out);
/* ---- locate / extract over the SA samples (FMIndex::loadSamples, locate and getSuffix of the reference's FMIndex) ----
 * A position is resolved by LF steps to the left until its suffix is sampled or starts a document (at most
 * sample rate - 1 steps).  The sample tables stay in HBM bit-packed, as the .sa file holds them.  Calling any of
 * the entry points below before samples are attached returns DSMFM_EINVAL; so do a position >= n, a document >= D,
 * and samples whose walks do not end within the longest document (an .sa file of another index).  Every call runs
 * on the searcher's stream and synchronises it. */
/* Attach the SA samples of THIS index: a `.sa` file (dsmfm_write_sa, or the reference's FMIndex::saveSamples),
 * or its bytes in memory (dsmfm_sa_serialize).  Replaces samples attached before. */
DSMFM_API int dsmfm_searcher_load_samples(dsmfm_searcher *s, const char *sa_path);
DSMFM_API int dsmfm_searcher_set_samples(dsmfm_searcher *s, const uint8_t *image, uint64_t bytes);
/* doc[k], offset[k] of the suffix at BWT position pos[k] (pos[k] < n) */
DSMFM_API int dsmfm_searcher_locate(dsmfm_searcher *s, const uint64_t *pos, uint64_t count, uint32_t *doc, uint64_t *offset);
DSMFM_API int dsmfm_searcher_locate_device(dsmfm_searcher *s, const void *pos_dev, uint64_t count, void *doc_dev, void *offset_dev);
/* every position of the intervals [sp[k], ep[k]] as dsmfm_searcher_count returns them (sp > ep: none); *total = their
 * number; total > cap -> DSMFM_ELIMIT and nothing but *total written */
DSMFM_API int dsmfm_searcher_locate_ranges(dsmfm_searcher *s, const uint64_t *sp, const uint64_t *ep, uint64_t count,
                                           uint64_t cap, uint32_t *doc, uint64_t *offset, uint64_t *total);
/* documents docs[k] (without terminator) at out[offsets[k] .. offsets[k+1]); offsets[0..count] always written;
 * offsets[count] > cap -> DSMFM_ELIMIT */
DSMFM_API int dsmfm_searcher_extract(dsmfm_searcher *s, const uint32_t *docs, uint64_t count, uint8_t *out, uint64_t cap,
                                     uint64_t *offsets);
/* Replaces: EnumerateQuery::enumerate (EnumerateQuery.cpp:9-37) with nextEnforced / nextSymbol (151-290), pushChar /
 * leftChar (39-103) and the encoding of ClientSocket::putc / putulong (ClientSocket.h:12-39) -- the mining client's
 * walk of the trie of all substrings that occur at least fmin times below `enforce_path`, SURVEY 8(f) row 4.  The
 * walk runs level by level on the GPU (one thread per node and symbol); the bytes are the reference's, in its
 * depth-first order: node := '(' sym node* freq ['R' count] leftChar ')' (Appendix B of SURVEY.md), i.e. exactly
 * what metaenumerate sends a metaserver after the handshake 'S' name '.' (metaenumerate.cpp:285-286), which the
 * caller writes itself.  maxdepth 0 = unlimited.  fmin >= 2 (with fmin 1 the reference follows unary paths symbol
 * by symbol, EnumerateQuery.cpp:105-149: not rebuilt).
 *   _fd: the stream is written to a file descriptor (a connected socket: the drop-in for ClientSocket);
 *   the other form returns it in memory (release with dsmfm_stream_free). */
DSMFM_API int dsmfm_searcher_enumerate_fd(dsmfm_searcher *s, const char *enforce_path, uint64_t fmin, uint32_t maxdepth, int fd,
                                          uint64_t *bytes_written);
DSMFM_API int dsmfm_searcher_enumerate(dsmfm_searcher *s, const char *enforce_path, uint64_t fmin, uint32_t maxdepth, uint8_t **out,
                                       uint64_t *out_bytes);
DSMFM_API void dsmfm_stream_free(uint8_t *p);
DSMFM_API const char *dsmfm_searcher_last_error(const dsmfm_searcher *s);
DSMFM_API void dsmfm_searcher_destroy(dsmfm_searcher *s);

/* Page-locked host memory (cudaHostAlloc) for the buffers handed to dsmfm_append_batch / dsmfm_append_fasta:
 * host-to-device copies from it run at the full PCIe rate.  NULL on failure. */
DSMFM_API void *dsmfm_alloc_pinned(size_t bytes);
DSMFM_API void dsmfm_free_pinned(void *p);

/* ---- kernel-level entry points used by the unit tests (host buffers in/out) ---- */

/* With DSMFM_GUARD=1 in the environment every device buffer of a builder carries 4 KB of pattern in front and
 * behind, checked when it is released: the number of buffers found overwritten so far (0 = clean). */
DSMFM_API uint64_t dsmfm_dbg_guard_violations(void);

/* Stable LSD radix sort of (key, value) pairs on bits [begin_bit, end_bit) with
 * the same onesweep kernels the build uses.  Sorts in place. */
DSMFM_API int dsmfm_dbg_radix_sort(int device, uint64_t *keys, uint32_t *vals, uint64_t n, int begin_bit, int end_bit);

/* The initial suffix sort of an unsharded build, stopped after the group heads: the build's code map, first-key
 * rule (first_key_bits <= 0: the default, else that many key bits), pack, keys with their digit counts, radix sort
 * and heads.  `docs` holds n bytes of '\0'-terminated, non-empty documents (n < 2^32 - 2112).  With ncuts > 0 the
 * text is packed and keyed word range by word range, as a batch streaming in from the host is: word_cuts are
 * increasing word indices in (0, words of the text).
 * Out (host): keys[n] (unsorted, text order), hist[8 * 256] (digit counts per 8-bit pass), sorted_keys[n], sa[n],
 * head[ceil(n/32)], remaining (ranks in groups of >= 2), bits per symbol, first_syms, carry (1: the BWT symbol
 * rides above the key; then diff[ceil(n/32)] and bwt[n] are written, else they are left untouched).
 * DSMFM_EINVAL (nothing launched) on malformed input. */
DSMFM_API int dsmfm_dbg_initial_sort(int device, const uint8_t *docs, uint64_t n, int first_key_bits,
                                     const uint64_t *word_cuts, uint32_t ncuts, uint64_t *keys, uint64_t *hist,
                                     uint64_t *sorted_keys, uint32_t *sa, uint32_t *head, uint32_t *diff, uint8_t *bwt,
                                     uint64_t *remaining, int *bits, int *first_syms, int *carry);

/* Wavelet tree + BitRank directories for an arbitrary byte sequence (the
 * HuffWT::makeHuffWT path alone); `out` pointers are valid until
 * dsmfm_dbg_free_index. */
DSMFM_API int dsmfm_dbg_wavelet(int device, const uint8_t *seq, uint64_t n, dsmfm_index *out, void **owner);
DSMFM_API void dsmfm_dbg_free_index(void *owner);

#ifdef __cplusplus
}
#endif
#endif /* DSMFM_H_ */
