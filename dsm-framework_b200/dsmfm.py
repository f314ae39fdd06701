"""ctypes binding of the C ABI in include/dsmfm.h (libdsmfm.so).

This is plumbing for the tests and bench.py; the product is the shared library
and the C++ facade in host/.  There is no CPU fallback: importing works
anywhere (so that symbol checks can run on a CPU-only box) but every call that
computes needs a B200 and fails loudly otherwise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSMFM_LIB") or os.path.join(_HERE, "libdsmfm.so")  # (DSMFM_LIB: a variant build, for A/B measurements)

OK, EINVAL, ECUDA, ENOMEM, EEMPTY, ELIMIT, EIO = 0, -1, -2, -3, -4, -5, -6
FLAG_KEEP_BWT, FLAG_KEEP_SA, FLAG_DEFAULT_STREAM = 1, 2, 4


class Options(C.Structure):
    _fields_ = [("device", C.c_int32), ("samplerate", C.c_uint32), ("expected_bytes", C.c_uint64),
                ("stream", C.c_void_p), ("flags", C.c_uint32), ("reserved", C.c_uint32),
                ("shard_index", C.c_uint32), ("shard_count", C.c_uint32), ("shard_span", C.c_uint32),
                ("reserved2", C.c_uint32)]


class Shard(C.Structure):
    _fields_ = [("n_total", C.c_uint64), ("rank_begin", C.c_uint64), ("count", C.c_uint64),
                ("bwt_dev", C.c_void_p), ("sa_dev", C.c_void_p)]


MAX_BLOCKS = 64


class BlockInfo(C.Structure):
    _fields_ = [("counts", C.c_uint64 * 256), ("bytes", C.c_uint64), ("documents", C.c_uint64),
                ("max_text_length", C.c_uint64), ("empty_document", C.c_uint32), ("reserved", C.c_uint32)]


class TextPlan(C.Structure):
    _fields_ = [("world", C.c_uint32), ("bits", C.c_uint32), ("n", C.c_uint64), ("documents", C.c_uint64),
                ("max_text_length", C.c_uint64), ("slot_words", C.c_uint64), ("text_bytes", C.c_uint64),
                ("counts", C.c_uint64 * 256), ("block_bytes", C.c_uint64 * MAX_BLOCKS)]


class PieceEdge(C.Structure):
    _fields_ = [("count", C.c_uint64), ("first_word", C.c_uint64), ("first", C.c_uint64 * 4), ("last_word", C.c_uint64),
                ("last", C.c_uint64 * 4), ("ch", C.c_uint64)]


class Piece(C.Structure):
    _fields_ = [("node", C.c_uint32), ("reserved", C.c_uint32), ("word_first", C.c_uint64), ("word_count", C.c_uint64),
                ("rs_first", C.c_uint64), ("rs_count", C.c_uint64), ("rb_first", C.c_uint64), ("rb_count", C.c_uint64),
                ("data", C.POINTER(C.c_uint64)), ("Rs", C.POINTER(C.c_uint64)), ("Rb", C.POINTER(C.c_uint8))]


class Pieces(C.Structure):
    _fields_ = [("n_internal", C.c_uint32), ("world", C.c_uint32), ("rank", C.c_uint32), ("reserved", C.c_uint32),
                ("bytes", C.c_uint64), ("piece", C.POINTER(Piece)), ("edge", C.POINTER(PieceEdge))]


class SaInfo(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("ends", C.c_uint64), ("documents", C.c_uint64)]


SA_VECTORS = 5


class Code(C.Structure):
    _fields_ = [("count", C.c_uint64), ("bits", C.c_uint32), ("code", C.c_uint32)]


class Node(C.Structure):
    _fields_ = [("leaf", C.c_uint8), ("ch", C.c_uint8), ("pad", C.c_uint8 * 6), ("nbits", C.c_uint64),
                ("integers", C.c_uint64), ("data", C.POINTER(C.c_uint64)), ("Rs", C.POINTER(C.c_uint64)),
                ("Rb", C.POINTER(C.c_uint8))]


class Index(C.Structure):
    _fields_ = [("n", C.c_uint64), ("samplerate", C.c_uint32), ("number_of_texts", C.c_uint32),
                ("max_text_length", C.c_uint64), ("C", C.c_uint64 * 256), ("codetable", Code * 256),
                ("n_nodes", C.c_uint32), ("reserved", C.c_uint32), ("nodes", C.POINTER(Node)),
                ("bwt", C.POINTER(C.c_uint8))]


class Stats(C.Structure):
    _fields_ = [("n", C.c_uint64), ("bases", C.c_uint64), ("bits_per_symbol", C.c_uint32), ("sigma", C.c_uint32),
                ("rounds", C.c_uint32), ("kernel_launches", C.c_uint32), ("active", C.c_uint64 * 32),
                ("fallback_elems", C.c_uint64), ("ms_total", C.c_float), ("ms_pack", C.c_float),
                ("ms_sort", C.c_float), ("ms_sort_pass", C.c_float), ("ms_refine", C.c_float), ("ms_bwt", C.c_float),
                ("ms_wt", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float), ("sort_passes", C.c_uint32),
                ("sort_launches", C.c_uint32), ("sort_pass_bytes", C.c_uint64), ("device_bytes_peak", C.c_uint64),
                ("ms_wall_build", C.c_float), ("ms_wall_fetch", C.c_float), ("ms_wall_alloc", C.c_float),
                ("streamed", C.c_uint32), ("refine_key_fetches", C.c_uint64), ("refine_launches", C.c_uint64),
                ("refine_members", C.c_uint64)]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d


class FastaInfo(C.Structure):
    _fields_ = [("consumed", C.c_uint64), ("records", C.c_uint64), ("documents", C.c_uint64), ("bases", C.c_uint64),
                ("doc_bytes", C.c_uint64), ("invalid_records", C.c_uint64), ("first_invalid_offset", C.c_uint64),
                ("bad_headers", C.c_uint64)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class DsmfmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("dsmfm error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """Load libdsmfm.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libdsmfm.so is missing (%s): build it with `make -C dsm-framework_b200` or "
                           "__graft_entry__.build(); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    B = C.c_void_p
    L.dsmfm_version.restype = C.c_int
    L.dsmfm_create.argtypes = [C.POINTER(Options), C.POINTER(B)]
    L.dsmfm_append.argtypes = [B, C.c_void_p, C.c_size_t]
    L.dsmfm_append_batch.argtypes = [B, C.c_void_p, C.c_size_t]
    L.dsmfm_append_batch_device.argtypes = [B, C.c_void_p, C.c_size_t]
    L.dsmfm_append_fasta.argtypes = [B, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(FastaInfo)]
    L.dsmfm_finish.argtypes = [B, C.POINTER(Index)]
    L.dsmfm_build_device.argtypes = [B]
    L.dsmfm_fetch.argtypes = [B, C.POINTER(Index)]
    L.dsmfm_write_fmi.argtypes = [C.POINTER(Index), C.c_char_p]
    L.dsmfm_fmi_size.argtypes = [C.POINTER(Index)]
    L.dsmfm_fmi_size.restype = C.c_uint64
    L.dsmfm_fmi_serialize.argtypes = [C.POINTER(Index), C.c_void_p, C.c_uint64]
    L.dsmfm_copy_sa.argtypes = [B, C.c_void_p, C.c_uint64, C.c_uint64]
    L.dsmfm_get_stats.argtypes = [B, C.POINTER(Stats)]
    L.dsmfm_last_error.argtypes = [B]
    L.dsmfm_last_error.restype = C.c_char_p
    L.dsmfm_destroy.argtypes = [B]
    L.dsmfm_destroy.restype = None
    L.dsmfm_release_cached.argtypes = [C.c_int]
    L.dsmfm_shard_info.argtypes = [B, C.POINTER(Shard)]
    L.dsmfm_assemble.argtypes = [B, C.c_void_p, C.c_uint64]
    L.dsmfm_shard_export.argtypes = [B, C.c_void_p, C.c_void_p]
    L.dsmfm_write_sa.argtypes = [B, C.c_char_p]
    L.dsmfm_sa_size.argtypes = [B]
    L.dsmfm_sa_size.restype = C.c_uint64
    L.dsmfm_sa_serialize.argtypes = [B, C.c_void_p, C.c_uint64]
    L.dsmfm_slice_hist.argtypes = [B, C.c_void_p]
    L.dsmfm_pieces_bytes.argtypes = [B, C.c_void_p, C.c_uint32, C.c_uint32]
    L.dsmfm_pieces_bytes.restype = C.c_uint64
    L.dsmfm_build_pieces.argtypes = [B, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    L.dsmfm_assemble_pieces.argtypes = [B, C.c_void_p, C.c_uint32, C.c_void_p]
    L.dsmfm_block_stats.argtypes = [B, C.POINTER(BlockInfo)]
    L.dsmfm_text_plan_make.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(TextPlan)]
    L.dsmfm_block_pack.argtypes = [B, C.POINTER(TextPlan), C.c_uint32, C.c_void_p, C.c_void_p]
    L.dsmfm_build_packed.argtypes = [B, C.POINTER(TextPlan), C.c_void_p, C.c_void_p]
    L.dsmfm_pieces_build.argtypes = [B, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(Pieces)]
    L.dsmfm_pieces_fetch.argtypes = [B, C.POINTER(Pieces)]
    L.dsmfm_pieces_merge.argtypes = [B, C.c_void_p, C.c_uint32]
    L.dsmfm_pieces_index.argtypes = [B, C.POINTER(Index)]
    L.dsmfm_pieces_write.argtypes = [B, C.c_char_p, C.c_int]
    L.dsmfm_sa_slice_info.argtypes = [B, C.POINTER(SaInfo)]
    L.dsmfm_sa_pieces_build.argtypes = [B, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    L.dsmfm_sa_pieces_merge.argtypes = [B, C.c_void_p, C.c_uint32]
    L.dsmfm_sa_pieces_write.argtypes = [B, C.c_char_p, C.c_int]
    S = C.c_void_p
    L.dsmfm_searcher_create.argtypes = [C.c_int, C.POINTER(Index), C.POINTER(S)]
    L.dsmfm_searcher_open.argtypes = [C.c_int, C.c_char_p, C.POINTER(S)]
    L.dsmfm_searcher_length.argtypes = [S]
    L.dsmfm_searcher_length.restype = C.c_uint64
    L.dsmfm_searcher_rank.argtypes = [S, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.dsmfm_searcher_lf.argtypes = [S, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.dsmfm_searcher_lf_device.argtypes = [S, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.dsmfm_searcher_access.argtypes = [S, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.dsmfm_searcher_extend.argtypes = [S, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.dsmfm_searcher_count.argtypes = [S, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.dsmfm_searcher_load_samples.argtypes = [S, C.c_char_p]
    L.dsmfm_searcher_set_samples.argtypes = [S, C.c_void_p, C.c_uint64]
    L.dsmfm_searcher_locate.argtypes = [S, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.dsmfm_searcher_locate_device.argtypes = [S, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.dsmfm_searcher_locate_ranges.argtypes = [S, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                               C.POINTER(C.c_uint64)]
    L.dsmfm_searcher_extract.argtypes = [S, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
    L.dsmfm_searcher_enumerate.argtypes = [S, C.c_char_p, C.c_uint64, C.c_uint32, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_uint64)]
    L.dsmfm_searcher_enumerate_fd.argtypes = [S, C.c_char_p, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(C.c_uint64)]
    L.dsmfm_stream_free.argtypes = [C.POINTER(C.c_uint8)]
    L.dsmfm_stream_free.restype = None
    L.dsmfm_searcher_last_error.argtypes = [S]
    L.dsmfm_searcher_last_error.restype = C.c_char_p
    L.dsmfm_searcher_destroy.argtypes = [S]
    L.dsmfm_searcher_destroy.restype = None
    L.dsmfm_dbg_guard_violations.restype = C.c_uint64
    L.dsmfm_dbg_radix_sort.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int]
    L.dsmfm_dbg_initial_sort.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint32] + \
        [C.c_void_p] * 8 + [C.POINTER(C.c_int)] * 3
    L.dsmfm_dbg_wavelet.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.POINTER(Index), C.POINTER(C.c_void_p)]
    L.dsmfm_dbg_free_index.argtypes = [C.c_void_p]
    L.dsmfm_dbg_free_index.restype = None
    _lib = L
    return L


def _ptr(buf):
    """(address, nbytes, keepalive) of bytes / bytearray / numpy array / torch tensor."""
    if isinstance(buf, (bytes, bytearray)):
        arr = (C.c_char * len(buf)).from_buffer_copy(buf) if isinstance(buf, bytes) else (C.c_char * len(buf)).from_buffer(buf)
        return C.addressof(arr), len(buf), arr
    if hasattr(buf, "data_ptr"):  # torch tensor (host or device)
        return buf.data_ptr(), buf.numel() * buf.element_size(), buf
    if hasattr(buf, "ctypes"):  # numpy
        return buf.ctypes.data, buf.nbytes, buf
    raise TypeError("unsupported buffer type %r" % type(buf))


def fmi_bytes(index):
    """Serialise a dsmfm_index into the bytes of the reference's .fmi file."""
    L = lib()
    size = L.dsmfm_fmi_size(C.byref(index))
    out = bytearray(size)
    arr = (C.c_char * size).from_buffer(out)
    rc = L.dsmfm_fmi_serialize(C.byref(index), C.addressof(arr), size)
    if rc != OK:
        raise DsmfmError(rc, "dsmfm_fmi_serialize failed")
    del arr
    return bytes(out)


class Builder:
    """Mirror of the reference's TextCollectionBuilder over the C ABI."""

    def __init__(self, device=-1, samplerate=0, expected_bytes=0, stream=None, flags=0, shard_index=0, shard_count=1,
                 shard_span=1):
        self._L = lib()
        opt = Options(device=device, samplerate=samplerate, expected_bytes=expected_bytes,
                      stream=stream, flags=flags, reserved=0, shard_index=shard_index, shard_count=shard_count,
                      shard_span=shard_span, reserved2=0)
        self._h = C.c_void_p()
        rc = self._L.dsmfm_create(C.byref(opt), C.byref(self._h))
        if rc != OK:
            raise DsmfmError(rc, (self._L.dsmfm_last_error(None) or b"").decode())
        self.index = None
        self._keep = []

    def _check(self, rc):
        if rc != OK:
            raise DsmfmError(rc, (self._L.dsmfm_last_error(self._h) or b"").decode())

    def insert_text(self, doc):
        """TextCollectionBuilder::InsertText: one document, no terminator."""
        addr, n, keep = _ptr(doc)
        self._check(self._L.dsmfm_append(self._h, addr, n))

    def append_batch(self, docs):
        """'\\0'-terminated documents back to back, in host memory."""
        addr, n, keep = _ptr(docs)
        self._keep.append(keep)
        self._check(self._L.dsmfm_append_batch(self._h, addr, n))

    def append_batch_device(self, tensor):
        addr, n, keep = _ptr(tensor)
        self._keep.append(keep)
        self._check(self._L.dsmfm_append_batch_device(self._h, addr, n))

    def append_fasta(self, text, final=True):
        """FASTA bytes (host memory) -> documents, parsed and transformed on the GPU (the reference CLI's record
        loop, builder.cpp:203-262).  Returns the dsmfm_fasta_info fields as a dict."""
        addr, n, keep = _ptr(text)
        info = FastaInfo()
        self._check(self._L.dsmfm_append_fasta(self._h, addr, n, 1 if final else 0, C.byref(info)))
        return info.as_dict()

    def build_device(self):
        self._check(self._L.dsmfm_build_device(self._h))
        self._keep = []  # the build has synchronised its stream: the appended buffers have been consumed

    def shard_info(self):
        sh = Shard()
        self._check(self._L.dsmfm_shard_info(self._h, C.byref(sh)))
        return sh

    def shard_export(self, bwt_dst=None, sa_dst=None):
        """Copies the slice into CUDA tensors: bwt_dst uint8[count], sa_dst int64/uint64[count]."""
        self._check(self._L.dsmfm_shard_export(self._h, bwt_dst.data_ptr() if bwt_dst is not None else None,
                                               sa_dst.data_ptr() if sa_dst is not None else None))

    # ---- wavelet tree built by several GPUs (include/dsmfm.h) ----
    def slice_hist(self):
        """Byte histogram of this builder's BWT slice: numpy uint64[256]."""
        import numpy as np
        out = np.zeros(256, dtype=np.uint64)
        self._check(self._L.dsmfm_slice_hist(self._h, out.ctypes.data))
        return out

    @staticmethod
    def _hist_table(hist_all):
        import numpy as np
        h = np.ascontiguousarray(hist_all, dtype=np.uint64)
        assert h.ndim == 2 and h.shape[1] == 256
        return h

    def pieces_bytes(self, hist_all, rank):
        """Size of slice `rank`'s piece buffer (rank == number of slices: all of them together)."""
        h = self._hist_table(hist_all)
        return int(self._L.dsmfm_pieces_bytes(self._h, h.ctypes.data, h.shape[0], rank))

    def build_pieces(self, hist_all, rank, dst):
        h = self._hist_table(hist_all)
        self._check(self._L.dsmfm_build_pieces(self._h, h.ctypes.data, h.shape[0], rank, dst.data_ptr()))

    def assemble_pieces(self, hist_all, pieces):
        h = self._hist_table(hist_all)
        self._keep.append(pieces)
        self._check(self._L.dsmfm_assemble_pieces(self._h, h.ctypes.data, h.shape[0], pieces.data_ptr()))

    # ---- packed-text exchange between builders (include/dsmfm.h, "one collection over several GPUs") ----
    def block_stats(self):
        """Statistics of this builder's block of documents as bytes (a dsmfm_block_info record, to be all-gathered)."""
        info = BlockInfo()
        self._check(self._L.dsmfm_block_stats(self._h, C.byref(info)))
        self._keep = []  # the stream has been synchronised: appended buffers are consumed
        return bytes(info)

    def block_pack(self, plan, rank, text):
        """Packs the block into slot `rank` of `text` (uint8 CUDA tensor of plan.text_bytes); returns the block's
        histogram of the top 12 key bits (numpy uint64[4096])."""
        import numpy as np
        top = np.zeros(4096, dtype=np.uint64)
        self._check(self._L.dsmfm_block_pack(self._h, C.byref(plan), rank, text.data_ptr(), top.ctypes.data))
        return top

    def build_packed(self, plan, text, top_sum):
        import numpy as np
        top = np.ascontiguousarray(top_sum, dtype=np.uint64)
        self._check(self._L.dsmfm_build_packed(self._h, C.byref(plan), text.data_ptr(), top.ctypes.data))

    def pieces_build(self, hist_all, rank, fetch=True):
        """Returns (Pieces, edges) -- edges: this builder's dsmfm_piece_edge records as bytes; (None, None) with
        fetch=False (the sections then stay in HBM until pieces_fetch)."""
        h = self._hist_table(hist_all)
        out = Pieces()
        self._check(self._L.dsmfm_pieces_build(self._h, h.ctypes.data, h.shape[0], rank, C.byref(out) if fetch else None))
        if not fetch:
            return None, None
        self.pieces = out
        return out, C.string_at(out.edge, C.sizeof(PieceEdge) * out.n_internal)

    def pieces_fetch(self):
        out = Pieces()
        self._check(self._L.dsmfm_pieces_fetch(self._h, C.byref(out)))
        self.pieces = out
        return out, C.string_at(out.edge, C.sizeof(PieceEdge) * out.n_internal)

    def pieces_merge(self, edges_all, world):
        """edges_all: the records of every builder in slice order, back to back (bytes)."""
        buf = C.create_string_buffer(bytes(edges_all), len(edges_all))
        self._check(self._L.dsmfm_pieces_merge(self._h, buf, world))

    def pieces_index(self):
        idx = Index()
        self._check(self._L.dsmfm_pieces_index(self._h, C.byref(idx)))
        return idx

    def pieces_write(self, prefix, header):
        self._check(self._L.dsmfm_pieces_write(self._h, os.fsencode(prefix), 1 if header else 0))

    # ---- .sa samples of a packed-text build (FLAG_KEEP_SA; include/dsmfm.h steps 8-11) ----
    def sa_slice_info(self):
        """This builder's dsmfm_sa_info record as bytes (to be all-gathered)."""
        info = SaInfo()
        self._check(self._L.dsmfm_sa_slice_info(self._h, C.byref(info)))
        return bytes(info)

    def sa_pieces_build(self, infos_all, world, rank):
        """infos_all: the records of every builder in slice order, back to back (bytes).  Returns this builder's
        SA_VECTORS dsmfm_piece_edge records as bytes."""
        buf = C.create_string_buffer(bytes(infos_all), len(infos_all))
        edges = (PieceEdge * SA_VECTORS)()
        self._check(self._L.dsmfm_sa_pieces_build(self._h, buf, world, rank, C.addressof(edges)))
        return bytes(edges)

    def sa_pieces_merge(self, edges_all, world):
        buf = C.create_string_buffer(bytes(edges_all), len(edges_all))
        self._check(self._L.dsmfm_sa_pieces_merge(self._h, buf, world))

    def sa_pieces_write(self, prefix, header):
        self._check(self._L.dsmfm_sa_pieces_write(self._h, os.fsencode(prefix), 1 if header else 0))

    def assemble(self, bwt_dev, n_total):
        """bwt_dev: device address (int) or torch CUDA tensor holding the concatenated BWT."""
        addr = bwt_dev.data_ptr() if hasattr(bwt_dev, "data_ptr") else int(bwt_dev)
        self._keep.append(bwt_dev)
        self._check(self._L.dsmfm_assemble(self._h, addr, n_total))

    def fetch(self):
        idx = Index()
        self._check(self._L.dsmfm_fetch(self._h, C.byref(idx)))
        self.index = idx
        return idx

    def finish(self):
        """TextCollectionBuilder::InitTextCollection."""
        idx = Index()
        self._check(self._L.dsmfm_finish(self._h, C.byref(idx)))
        self.index = idx
        self._keep = []
        return idx

    def fmi(self):
        return fmi_bytes(self.index)

    def bwt(self):
        if not self.index or not self.index.bwt:
            raise RuntimeError("build with FLAG_KEEP_BWT")
        return C.string_at(self.index.bwt, self.index.n)

    def suffix_array(self, first=0, count=None):
        import numpy as np
        if count is None:
            count = self.index.n - first
        out = np.empty(count, dtype=np.uint32)
        self._check(self._L.dsmfm_copy_sa(self._h, out.ctypes.data, first, count))
        return out

    def save(self, prefix):
        rc = self._L.dsmfm_write_fmi(C.byref(self.index), os.fsencode(prefix))
        if rc != OK:
            raise DsmfmError(rc, "dsmfm_write_fmi failed")

    def sa_file(self):
        """Bytes of the `.sa` file (FMIndex::saveSamples); needs FLAG_KEEP_SA."""
        size = self._L.dsmfm_sa_size(self._h)
        if size == 0:
            raise DsmfmError(EINVAL, (self._L.dsmfm_last_error(self._h) or b"").decode())
        out = bytearray(size)
        arr = (C.c_char * size).from_buffer(out)
        self._check(self._L.dsmfm_sa_serialize(self._h, C.addressof(arr), size))
        del arr
        return bytes(out)

    def save_samples(self, prefix):
        """TextCollection::saveSamples: writes <prefix>.sa"""
        self._check(self._L.dsmfm_write_sa(self._h, os.fsencode(prefix)))

    def stats(self):
        s = Stats()
        self._check(self._L.dsmfm_get_stats(self._h, C.byref(s)))
        return s

    def close(self):
        if self._h:
            self._L.dsmfm_destroy(self._h)
            self._h = C.c_void_p()
            self.index = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Searcher:
    """The query half of an index on the GPU: batched FMIndex::LF / getL / interval extension (include/dsmfm.h)."""

    def __init__(self, source, device=0):
        """source: path of an .fmi file, or a Builder that has finished (its sections are uploaded)."""
        import numpy as np
        self._np = np
        self._L = lib()
        self._h = C.c_void_p()
        if isinstance(source, (str, bytes, os.PathLike)):
            rc = self._L.dsmfm_searcher_open(device, os.fsencode(source), C.byref(self._h))
        else:
            rc = self._L.dsmfm_searcher_create(device, C.byref(source.index), C.byref(self._h))
        if rc != OK:
            raise DsmfmError(rc, (self._L.dsmfm_searcher_last_error(None) or b"").decode())
        self.n = self._L.dsmfm_searcher_length(self._h)

    def _check(self, rc):
        if rc != OK:
            raise DsmfmError(rc, (self._L.dsmfm_searcher_last_error(self._h) or b"").decode())

    def _ci(self, c, i):
        np = self._np
        i = np.ascontiguousarray(np.asarray(i, dtype=np.uint64))
        c = np.ascontiguousarray(np.broadcast_to(np.asarray(c, dtype=np.uint8), i.shape))
        return c, i, np.empty(i.shape, dtype=np.uint64)

    def rank(self, c, i):
        c, i, out = self._ci(c, i)
        self._check(self._L.dsmfm_searcher_rank(self._h, c.ctypes.data, i.ctypes.data, out.ctypes.data, i.size))
        return out

    def lf(self, c, i):
        c, i, out = self._ci(c, i)
        self._check(self._L.dsmfm_searcher_lf(self._h, c.ctypes.data, i.ctypes.data, out.ctypes.data, i.size))
        return out

    def lf_device(self, c, i, out):
        """torch tensors on the searcher's device: uint8 [count], int64/uint64 [count], int64/uint64 [count]"""
        self._check(self._L.dsmfm_searcher_lf_device(self._h, c.data_ptr(), i.data_ptr(), out.data_ptr(), i.numel()))

    def access(self, i):
        np = self._np
        i = np.ascontiguousarray(np.asarray(i, dtype=np.uint64))
        sym, rank = np.empty(i.shape, dtype=np.uint8), np.empty(i.shape, dtype=np.uint64)
        self._check(self._L.dsmfm_searcher_access(self._h, i.ctypes.data, sym.ctypes.data, rank.ctypes.data, i.size))
        return sym, rank

    def extend(self, sp, ep, symbols=b"ACGT"):
        np = self._np
        sp = np.ascontiguousarray(np.asarray(sp, dtype=np.uint64))
        ep = np.ascontiguousarray(np.asarray(ep, dtype=np.uint64))
        sym = np.frombuffer(bytes(symbols), dtype=np.uint8)
        so, eo = np.empty((sp.size, sym.size), dtype=np.uint64), np.empty((sp.size, sym.size), dtype=np.uint64)
        self._check(self._L.dsmfm_searcher_extend(self._h, sp.ctypes.data, ep.ctypes.data, sp.size, sym.ctypes.data,
                                                  sym.size, so.ctypes.data, eo.ctypes.data))
        return so, eo

    def count(self, patterns):
        """patterns: list of bytes -> (sp, ep) arrays; the pattern occurs ep - sp + 1 times if sp <= ep"""
        np = self._np
        off = np.zeros(len(patterns) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(p) for p in patterns])
        blob = np.frombuffer(b"".join(patterns) + b"\0", dtype=np.uint8)
        sp, ep = np.empty(len(patterns), dtype=np.uint64), np.empty(len(patterns), dtype=np.uint64)
        self._check(self._L.dsmfm_searcher_count(self._h, blob.ctypes.data, off.ctypes.data, len(patterns),
                                                 sp.ctypes.data, ep.ctypes.data))
        return sp, ep

    # ---- locate / extract over the SA samples (include/dsmfm.h) ----
    def load_samples(self, source):
        """source: path of an .sa file, or its bytes (Builder.sa_file()).  Replaces samples attached before."""
        if isinstance(source, (bytes, bytearray, memoryview)):
            img = self._np.frombuffer(bytes(source), dtype=self._np.uint8)
            self._check(self._L.dsmfm_searcher_set_samples(self._h, img.ctypes.data if img.size else None, img.size))
        else:
            self._check(self._L.dsmfm_searcher_load_samples(self._h, os.fsencode(source)))

    def locate(self, pos):
        """BWT positions -> (document uint32, offset in the document uint64)"""
        np = self._np
        pos = np.ascontiguousarray(np.asarray(pos, dtype=np.uint64))
        doc, off = np.empty(pos.shape, dtype=np.uint32), np.empty(pos.shape, dtype=np.uint64)
        self._check(self._L.dsmfm_searcher_locate(self._h, pos.ctypes.data, pos.size, doc.ctypes.data, off.ctypes.data))
        return doc, off

    def locate_device(self, pos, doc, offset):
        """torch tensors on the searcher's device: int64/uint64 [count] in, int32/uint32 [count] and int64/uint64 [count] out"""
        for t, name, dtypes in ((pos, "pos", ("torch.int64", "torch.uint64")), (doc, "doc", ("torch.int32", "torch.uint32")),
                                (offset, "offset", ("torch.int64", "torch.uint64"))):
            if str(t.dtype) not in dtypes or not t.is_cuda or not t.is_contiguous() or t.numel() != pos.numel():
                raise ValueError("locate_device: %s must be a contiguous CUDA tensor of %d %s entries, got %s %s on %s"
                                 % (name, pos.numel(), " / ".join(dtypes), tuple(t.shape), t.dtype, t.device))
        self._check(self._L.dsmfm_searcher_locate_device(self._h, pos.data_ptr(), pos.numel(), doc.data_ptr(), offset.data_ptr()))

    def locate_ranges(self, sp, ep):
        """Every position of the intervals [sp[k], ep[k]] (sp > ep: none) -> (doc, offset, starts): interval k's
        occurrences are doc / offset[starts[k]:starts[k+1]], in BWT order."""
        np = self._np
        sp = np.ascontiguousarray(np.asarray(sp, dtype=np.uint64))
        ep = np.ascontiguousarray(np.asarray(ep, dtype=np.uint64))
        sizes = np.where(sp <= ep, ep - sp + np.uint64(1), np.uint64(0))
        starts = np.zeros(sp.size + 1, dtype=np.uint64)
        starts[1:] = np.cumsum(sizes, dtype=np.uint64)
        cap = int(starts[-1])
        doc, off = np.empty(cap, dtype=np.uint32), np.empty(cap, dtype=np.uint64)
        total = C.c_uint64()
        self._check(self._L.dsmfm_searcher_locate_ranges(self._h, sp.ctypes.data, ep.ctypes.data, sp.size, cap, doc.ctypes.data,
                                                         off.ctypes.data, C.byref(total)))
        return doc, off, starts

    def extract(self, docs):
        """Document ids -> list of their bytes (without terminator)."""
        np = self._np
        docs = np.ascontiguousarray(np.asarray(docs, dtype=np.uint32))
        offsets = np.empty(docs.size + 1, dtype=np.uint64)
        rc = self._L.dsmfm_searcher_extract(self._h, docs.ctypes.data, docs.size, None, 0, offsets.ctypes.data)
        if rc != ELIMIT:
            self._check(rc)
        out = np.empty(int(offsets[-1]), dtype=np.uint8)
        self._check(self._L.dsmfm_searcher_extract(self._h, docs.ctypes.data, docs.size, out.ctypes.data, out.size,
                                                   offsets.ctypes.data))
        blob = out.tobytes()
        return [blob[offsets[k]:offsets[k + 1]] for k in range(docs.size)]

    def enumerate(self, enforce_path, fmin=10, maxdepth=0):
        """EnumerateQuery::enumerate: the client's byte stream (without the handshake) for the trie below enforce_path."""
        out, n = C.POINTER(C.c_uint8)(), C.c_uint64()
        self._check(self._L.dsmfm_searcher_enumerate(self._h, bytes(enforce_path), fmin, maxdepth, C.byref(out), C.byref(n)))
        try:
            return C.string_at(out, n.value)
        finally:
            self._L.dsmfm_stream_free(out)

    def enumerate_to_fd(self, enforce_path, fd, fmin=10, maxdepth=0):
        n = C.c_uint64()
        self._check(self._L.dsmfm_searcher_enumerate_fd(self._h, bytes(enforce_path), fmin, maxdepth, fd, C.byref(n)))
        return n.value

    def close(self):
        if self._h:
            self._L.dsmfm_searcher_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def text_plan(infos):
    """infos: list of dsmfm_block_info records (bytes) in block order -> dsmfm_text_plan (host arithmetic only)."""
    blob = b"".join(infos)
    world = len(infos)
    assert len(blob) == world * C.sizeof(BlockInfo)
    buf = C.create_string_buffer(blob, len(blob))
    plan = TextPlan()
    rc = lib().dsmfm_text_plan_make(buf, world, C.byref(plan))
    if rc != OK:
        raise DsmfmError(rc, "dsmfm_text_plan_make failed" + (" (a block holds an empty document)" if rc == EEMPTY else ""))
    return plan


def build_fmi(docs, **kw):
    """docs: '\\0'-terminated documents (bytes-like).  Returns the .fmi bytes."""
    with Builder(**kw) as b:
        if len(docs):
            b.append_batch(docs)
        b.finish()
        return b.fmi()


def radix_sort(keys, vals, begin_bit=0, end_bit=64, device=0):
    """In-place stable sort of numpy uint64 keys / uint32 vals with the build's one-sweep kernels."""
    L = lib()
    rc = L.dsmfm_dbg_radix_sort(device, keys.ctypes.data, vals.ctypes.data, keys.size, begin_bit, end_bit)
    if rc != OK:
        raise DsmfmError(rc, (L.dsmfm_last_error(None) or b"").decode())


def initial_sort(docs, first_key_bits=0, word_cuts=None, device=0):
    """The initial suffix sort of an unsharded build, up to the group heads (dsmfm_dbg_initial_sort).
    docs: numpy uint8 '\\0'-terminated documents.  Returns a dict of numpy arrays: keys, hist (8 x 256),
    sorted_keys, sa, head, diff, bwt (diff / bwt stay zero when carry == 0) and the ints remaining, bits,
    first_syms, carry."""
    import numpy as np
    L = lib()
    docs = np.ascontiguousarray(docs, dtype=np.uint8)
    n = docs.size
    cuts = np.ascontiguousarray(word_cuts if word_cuts is not None else [], dtype=np.uint64)
    hw = (n + 31) // 32
    out = dict(keys=np.empty(n, np.uint64), hist=np.zeros((8, 256), np.uint64), sorted_keys=np.empty(n, np.uint64),
               sa=np.empty(n, np.uint32), head=np.empty(hw, np.uint32), diff=np.zeros(hw, np.uint32),
               bwt=np.zeros(n, np.uint8), remaining=np.zeros(1, np.uint64))
    bits, first_syms, carry = C.c_int(), C.c_int(), C.c_int()
    rc = L.dsmfm_dbg_initial_sort(device, docs.ctypes.data, n, first_key_bits, cuts.ctypes.data if cuts.size else None,
                                  cuts.size, *[out[k].ctypes.data for k in ("keys", "hist", "sorted_keys", "sa", "head",
                                                                             "diff", "bwt", "remaining")],
                                  C.byref(bits), C.byref(first_syms), C.byref(carry))
    if rc != OK:
        raise DsmfmError(rc, (L.dsmfm_last_error(None) or b"").decode())
    out.update(remaining=int(out["remaining"][0]), bits=bits.value, first_syms=first_syms.value, carry=carry.value)
    return out


def wavelet_fmi(seq, device=0):
    """.fmi bytes of a wavelet tree built over an arbitrary byte sequence (numberOfTexts/maxTextLength = 0)."""
    L = lib()
    addr, n, keep = _ptr(seq)
    idx = Index()
    owner = C.c_void_p()
    rc = L.dsmfm_dbg_wavelet(device, addr, n, C.byref(idx), C.byref(owner))
    if rc != OK:
        raise DsmfmError(rc, (L.dsmfm_last_error(None) or b"").decode())
    try:
        return fmi_bytes(idx)
    finally:
        L.dsmfm_dbg_free_index(owner)
