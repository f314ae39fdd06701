"""One FM-index over reads held by several GPUs of one box (SURVEY.md section 8e; BASELINE.json configs[3]).

One process per GPU (torchrun).  Rank r holds a contiguous block of the documents (document ids are global:
all documents of rank r precede those of rank r+1, exactly as if they had been inserted one after the other
into one TextCollectionBuilder).  What replaces incbwt's batch merge by backward search
(incbwt/rlcsa_builder.cpp:245-318) is that the merged order is a property of the text alone:

  1. every rank takes the statistics of its block (histogram, documents, longest document); the records are
     all-gathered (2 KB each) and every rank derives the same plan: alphabet, bits per symbol, slot size;
  2. every rank packs ITS block (3 bits per symbol for reads) into its slot of the packed text and counts the
     top 12 key bits of its suffixes; the slots are all-gathered over NVLink (NCCL, in place: 0.375 bytes per
     symbol instead of the raw text's 1), the 4096-bin histograms are summed;
  3. every rank suffix-sorts ITS key ranges of the global suffix order (dsmfm_options.shard_*), selecting the
     suffixes from the replicated packed text -- the refinement keys come from the same text, so the sort
     needs no exchange at all -- and ends up with a contiguous slice of the global BWT;
  4. the slices' byte histograms are all-gathered (2 KB each): they fix, for every node of the Huffman-shaped
     wavelet tree, which bits of the node every slice contributes and how many ones precede them.  Every rank
     builds its share of every node -- bit words, Rs and Rb directories -- on its own GPU, copies it to its
     own host memory, and after an exchange of the few words next to the slice boundaries (96 bytes per node
     and rank) writes it straight into the `.fmi` file at the offsets of FMIndex::save's layout;
  5. with samples (engines whose builders keep the suffix array, dsmfm.FLAG_KEEP_SA): the same for the five bit
     vectors of the `.sa` file.  The ranks all-gather their slices' sample / end-marker / document counts (24 bytes
     each), which fix every rank's range of every vector; the rest is step 4 again.

No rank ever holds the whole index and nothing funnels through one GPU.  torch.distributed is plumbing only:
the phases below are explicit so that the same host logic runs (a) one rank per process over NCCL or gloo and
(b) all ranks in one process, one after the other, on a single GPU (tests on a one-GPU box).  `engine`
abstracts the device work; tests/cpu_engine.py is a numpy model of it for the gloo tests.
"""
import os
import time

import numpy as np
import torch


class CudaEngine:
    """The device work through the C ABI (libdsmfm.so), on an explicit stream: torch's collectives are issued
    with that stream current, so everything a rank does is ordered on ONE stream."""

    def __init__(self, device, flags=0, samplerate=0):
        import dsmfm
        self._dsmfm = dsmfm
        self.device = device
        self.flags = flags
        self.samplerate = samplerate
        with torch.cuda.device(device):
            self.stream = torch.cuda.Stream()

    def tensor_device(self):
        return torch.device("cuda", self.device)

    def stream_context(self):
        return torch.cuda.stream(self.stream)

    def open(self, local_docs, rank, world, ranges_per_gpu):
        k = max(1, int(ranges_per_gpu))
        b = self._dsmfm.Builder(device=self.device, stream=self.stream.cuda_stream, expected_bytes=local_docs.numel(),
                                flags=self.flags, samplerate=self.samplerate, shard_index=rank * k, shard_count=world * k,
                                shard_span=k)
        try:
            if local_docs.numel():
                if local_docs.is_cuda:
                    self.stream.wait_stream(torch.cuda.current_stream(local_docs.device))  # whoever produced it
                    b.append_batch_device(local_docs)
                else:
                    b.append_batch(local_docs)
        except Exception:
            b.close()
            raise
        return b

    def block_stats(self, b):
        return b.block_stats()

    def plan(self, infos):
        p = self._dsmfm.text_plan(infos)
        return p, int(p.text_bytes), int(p.slot_words) * 8

    def new_text(self, text_bytes):
        return torch.empty(text_bytes, dtype=torch.uint8, device=self.tensor_device())

    def block_pack(self, b, plan, rank, text):
        return b.block_pack(plan, rank, text)

    def build_packed(self, b, plan, text, top_sum):
        b.build_packed(plan, text, top_sum)
        info = b.shard_info()
        return int(info.rank_begin), int(info.count)

    def slice_hist(self, b):
        return b.slice_hist()

    def pieces_build(self, b, hist_all, rank, fetch=True):
        pieces, edges = b.pieces_build(hist_all, rank, fetch)
        return (edges, int(pieces.bytes)) if fetch else (None, 0)

    def pieces_merge(self, b, edges_all, world):
        b.pieces_merge(edges_all, world)

    def pieces_write(self, b, prefix, header):
        b.pieces_write(prefix, header)

    def sa_info(self, b):
        return b.sa_slice_info()

    def sa_pieces_build(self, b, infos_all, world, rank):
        return b.sa_pieces_build(infos_all, world, rank)

    def sa_pieces_merge(self, b, edges_all, world):
        b.sa_pieces_merge(edges_all, world)

    def sa_pieces_write(self, b, prefix, header):
        b.sa_pieces_write(prefix, header)

    def stats(self, b):
        return b.stats()

    def close(self, b):
        b.close()


def block_of(n_items, rank, world):
    """Contiguous block [begin, end) of n_items for `rank` of `world` (sizes differ by at most one)."""
    q, r = divmod(n_items, world)
    begin = rank * q + min(rank, r)
    return begin, begin + q + (1 if rank < r else 0)


def check_tiling(begins, counts, n_total):
    """The ranks' slices must tile the suffix order [0, n_total) in rank order, without gaps."""
    pos = 0
    for r, (b, c) in enumerate(zip(begins, counts)):
        if c and b != pos:
            raise RuntimeError("BWT slices do not tile the suffix order: rank %d begins at %d, expected %d" % (r, b, pos))
        pos += c
    if pos != n_total:
        raise RuntimeError("BWT slices cover %d of %d suffixes" % (pos, n_total))


class ShardedBuild:
    """One rank's share of the build as explicit phases; what travels between two phases is named in the
    docstring of the phase that produces it."""

    def __init__(self, engine, rank, world, ranges_per_gpu=1):
        self.engine, self.rank, self.world, self.ranges = engine, rank, world, ranges_per_gpu
        self.handle = None
        self.text = None
        self.marks = []
        self._t = time.perf_counter()

    def _mark(self, name):
        if os.environ.get("DSMFM_MG_TRACE"):
            if self.engine.tensor_device().type == "cuda":
                torch.cuda.synchronize()
            t = time.perf_counter()
            self.marks.append((name, 1000 * (t - self._t)))
            self._t = t

    def stats(self, local_docs):
        """-> this block's dsmfm_block_info record (all-gather them in rank order)."""
        self._t = time.perf_counter()
        self.handle = self.engine.open(local_docs, self.rank, self.world, self.ranges)
        info = self.engine.block_stats(self.handle)
        self._mark("stats")
        return info

    def pack(self, infos):
        """-> (text, slot_bytes, top): the packed text with THIS rank's slot filled (all-gather the slots in place)
        and the block's histogram of the top 12 key bits (sum them over the ranks)."""
        self.plan, text_bytes, self.slot_bytes = self.engine.plan(infos)
        self.n_total = int(self.plan.n)
        self.text = self.engine.new_text(text_bytes)
        top = self.engine.block_pack(self.handle, self.plan, self.rank, self.text)
        self._mark("pack")
        return self.text, self.slot_bytes, top

    def sort(self, top_sum):
        """-> (rank_begin, count, hist): this rank's slice of the global suffix order and the byte histogram of
        its BWT slice (all-gather all three)."""
        self._mark("exchange_text")
        self.rank_begin, self.count = self.engine.build_packed(self.handle, self.plan, self.text, top_sum)
        self.text = None  # the sort is done with it
        hist = self.engine.slice_hist(self.handle)
        if int(hist.sum()) != self.count:
            raise RuntimeError("slice histogram of rank %d does not match its slice" % self.rank)
        self._mark("sort")
        return self.rank_begin, self.count, hist

    def pieces(self, begins, counts, hist_all, fetch=True):
        """-> this rank's dsmfm_piece_edge records (all-gather them in rank order); None with fetch=False: the
        rank's share of the sections is built and stays in HBM (device-resident timing)."""
        check_tiling(begins, counts, self.n_total)
        self.hist_all = np.ascontiguousarray(hist_all, dtype=np.uint64).reshape(self.world, 256)
        if fetch:
            edges, self.section_bytes = self.engine.pieces_build(self.handle, self.hist_all, self.rank)
        else:
            edges, self.section_bytes = self.engine.pieces_build(self.handle, self.hist_all, self.rank, False)
        self._mark("pieces")
        return edges

    def merge(self, edges_all):
        self.engine.pieces_merge(self.handle, b"".join(edges_all), self.world)
        self._mark("merge")

    def write(self, prefix):
        """Every rank writes its share into <prefix>.fmi; rank 0 adds header, node table and tail."""
        self.engine.pieces_write(self.handle, prefix, self.rank == 0)

    def sample_info(self):
        """-> this rank's dsmfm_sa_info record: samples and end markers of its slice, documents of its block
        (all-gather them in rank order)."""
        return self.engine.sa_info(self.handle)

    def samples(self, infos_all):
        """-> this rank's dsmfm_piece_edge records of the five `.sa` vectors (all-gather them in rank order)."""
        edges = self.engine.sa_pieces_build(self.handle, b"".join(infos_all), self.world, self.rank)
        self._mark("samples")
        return edges

    def merge_samples(self, edges_all):
        self.engine.sa_pieces_merge(self.handle, b"".join(edges_all), self.world)

    def write_samples(self, prefix):
        """Every rank writes its share into <prefix>.sa; rank 0 adds the headers."""
        self.engine.sa_pieces_write(self.handle, prefix, self.rank == 0)

    def build_stats(self):
        return self.engine.stats(self.handle) if hasattr(self.engine, "stats") else None

    def report(self):
        import sys
        s = self.build_stats()
        extra = ""
        if s is not None:
            extra = " | build: sort %.1f refine %.1f wt %.1f total %.1f, wall %.1f of which alloc %.1f, count %d" % (
                s.ms_sort, s.ms_refine, s.ms_wt, s.ms_total, s.ms_wall_build, s.ms_wall_alloc, self.count)
        print("[multigpu rank %d] " % self.rank + " ".join("%s %.1f ms" % m for m in self.marks) + extra, file=sys.stderr)

    def close(self):
        if self.handle is not None:
            self.engine.close(self.handle)
            self.handle = None
        self.text = None


# ---- (a) one rank per process: torch.distributed ------------------------------------------------------------

def _all_gather_bytes(dist, record, device):
    """Fixed-size records (bytes) of every rank, in rank order."""
    world = dist.get_world_size()
    t = torch.frombuffer(bytearray(record), dtype=torch.uint8).to(device)
    out = torch.empty(world * t.numel(), dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(out, t)
    blob = out.cpu().numpy().tobytes()
    return [blob[i * len(record):(i + 1) * len(record)] for i in range(world)]


def _all_gather_u64(dist, values, device):
    """numpy uint64[k] of every rank -> uint64[world, k]."""
    a = np.ascontiguousarray(values, dtype=np.uint64)
    recs = _all_gather_bytes(dist, a.tobytes(), device)
    return np.stack([np.frombuffer(r, dtype=np.uint64) for r in recs])


def build_sharded(dist, local_docs, engine, ranges_per_gpu=1, fetch=True, samples=False):
    """Builds ONE index over the documents of all ranks (rank order = document order).

    local_docs: uint8 tensor (pinned host or device) with this rank's '\\0'-terminated documents.
    Returns the rank's ShardedBuild, merged: sb.write(prefix) puts the rank's share into the `.fmi` file,
    sb.section_bytes is what it holds in host memory.  fetch=False stops with every rank's share of the sections
    in its HBM (what a device-resident measurement times).  samples=True (the engine's builders keep the suffix
    array) also exchanges the `.sa` pieces: sb.write_samples(prefix) then writes the rank's share of <prefix>.sa.
    Close it when done."""
    world, rank = dist.get_world_size(), dist.get_rank()
    device = engine.tensor_device()
    sb = ShardedBuild(engine, rank, world, ranges_per_gpu)
    ctx = engine.stream_context() if hasattr(engine, "stream_context") else _Null()
    try:
        with ctx:
            infos = _all_gather_bytes(dist, sb.stats(local_docs), device)
            text, slot_bytes, top = sb.pack(infos)
            if world > 1:
                mine = text[rank * slot_bytes:(rank + 1) * slot_bytes]
                dist.all_gather_into_tensor(text[:world * slot_bytes], mine)  # in place, over NVLink
            top_sum = _all_gather_u64(dist, top, device).sum(axis=0, dtype=np.uint64)
            rank_begin, count, hist = sb.sort(top_sum)
            rec = _all_gather_u64(dist, np.concatenate([np.array([rank_begin, count], dtype=np.uint64), hist]), device)
            edges = sb.pieces([int(x) for x in rec[:, 0]], [int(x) for x in rec[:, 1]], rec[:, 2:], fetch)
            if fetch:
                sb.merge(_all_gather_bytes(dist, edges, device))
            if samples:
                sa_edges = sb.samples(_all_gather_bytes(dist, sb.sample_info(), device))
                sb.merge_samples(_all_gather_bytes(dist, sa_edges, device))
    except Exception:
        sb.close()
        raise
    if os.environ.get("DSMFM_MG_TRACE"):
        sb.report()
    return sb


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


# ---- (b) all ranks in one process, one after the other (one GPU, or the CPU model) ----------------------------

def build_sharded_local(blocks, engines, ranges_per_gpu=1, samples=False):
    """blocks[r]: uint8 tensor with rank r's documents; engines[r]: its engine (they may share a device).
    The exchanges of build_sharded become plain copies.  Returns the list of merged ShardedBuilds."""
    world = len(blocks)
    sbs = [ShardedBuild(engines[r], r, world, ranges_per_gpu) for r in range(world)]
    try:
        infos = [sb.stats(blocks[r]) for r, sb in enumerate(sbs)]
        packed = [sb.pack(infos) for sb in sbs]
        slot = packed[0][1]
        for r in range(world):  # the all-gather: everybody's slot into everybody's text
            for q in range(world):
                if q != r:
                    packed[q][0][r * slot:(r + 1) * slot].copy_(packed[r][0][r * slot:(r + 1) * slot])
        for e in engines:
            if e.tensor_device().type == "cuda":
                torch.cuda.synchronize(e.tensor_device())
        top_sum = np.sum(np.stack([p[2] for p in packed]), axis=0, dtype=np.uint64)
        del packed
        sorted_ = [sb.sort(top_sum) for sb in sbs]
        begins, counts = [s[0] for s in sorted_], [s[1] for s in sorted_]
        hist_all = np.stack([s[2] for s in sorted_])
        edges = [sb.pieces(begins, counts, hist_all) for sb in sbs]
        for sb in sbs:
            sb.merge(edges)
        if samples:
            infos = [sb.sample_info() for sb in sbs]
            sa_edges = [sb.samples(infos) for sb in sbs]
            for sb in sbs:
                sb.merge_samples(sa_edges)
    except Exception:
        for sb in sbs:
            sb.close()
        raise
    return sbs
