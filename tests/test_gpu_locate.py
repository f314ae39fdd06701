"""GPU suite: locate and extract over the SA samples of the `.sa` file (dsmfm_searcher_load_samples / locate /
locate_ranges / extract, csrc/search.cu).  The expected value is always the brute-force suffix array -- the oracle's
or the builder's -- and the documents themselves; the sample tables are only ever the input."""
import ctypes as C
import json
import os
import struct

import numpy as np
import pytest

import cases
import oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MANIFEST = json.load(open(os.path.join(GOLDEN, "manifest.json")))


def _golden(name):
    with open(os.path.join(GOLDEN, name), "rb") as f:
        return f.read()


def _doc_of(docs, sa):
    """(document, offset) of text positions `sa` in '\\0'-terminated documents"""
    text = np.frombuffer(bytes(docs), dtype=np.uint8)
    starts = np.concatenate([[0], np.flatnonzero(text == 0)[:-1] + 1]).astype(np.uint64)
    sa = np.asarray(sa, dtype=np.uint64)
    doc = np.searchsorted(starts, sa, side="right") - 1
    return doc.astype(np.uint32), sa - starts[doc]


def _sa_sections(img):
    """byte offset and (count, width) of the four BlockArrays of an .sa image"""
    n, integers = struct.unpack_from("<QQ", img, 0)
    pos = 24 + 8 * integers + 8 * (n // 256 + 1) + n // 64 + 1
    out = []
    for _ in range(4):
        count, width = struct.unpack_from("<QQ", img, pos)
        out.append((pos, count, width))
        pos += 16 + 8 * (count * width // 64 + 1)
    assert pos == len(img)
    return out


@pytest.mark.parametrize("fn", sorted(MANIFEST["sa"]))
def test_reference_samples_locate_every_position_and_extract_every_document(fn):
    """The reference's own .fmi / .sa pairs: every BWT position against the oracle's suffix array."""
    import dsmfm
    case = MANIFEST["sa"][fn]["case"]
    docs, nd = oracle.fasta_to_docs(_golden(case + ".fasta"))
    _, sa = oracle.bwt(docs, want_sa=True)
    with dsmfm.Searcher(os.path.join(GOLDEN, case + ".fmi")) as s:
        s.load_samples(os.path.join(GOLDEN, fn))
        doc, off = s.locate(np.arange(s.n, dtype=np.uint64))
        want_doc, want_off = _doc_of(docs, sa)
        assert np.array_equal(doc, want_doc) and np.array_equal(off, want_off)
        assert s.extract(np.arange(nd)) == bytes(docs).split(b"\0")[:-1]


def _dup_docs(seed):
    rng = np.random.default_rng(seed)
    reads = [bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=int(rng.integers(1, 40)))) for _ in range(20)]
    return b"".join(reads[int(i)] + b"\0" for i in rng.integers(0, len(reads), size=300))


def _docs_of(kind):
    if kind == "dup":
        return _dup_docs(7)
    alpha = {"acgt": "ACGT", "colour": "ACGT0123.", "polya": "A"}[kind]
    return oracle.fasta_to_docs(cases.rnd_fasta(51, 300, 60, alpha=alpha, genome=800))[0]


@pytest.mark.parametrize("kind", ["acgt", "colour", "polya", "dup"])
@pytest.mark.parametrize("rate", [1, 2, 7, 124, "above"])
def test_built_index_locates_like_its_suffix_array(kind, rate, tmp_path):
    """Rate 1: every walk is 0 steps.  Above the longest document: no samples, every walk ends at a document start.
    Samples from sa_file() bytes and from save_samples -> load_samples answer identically."""
    import dsmfm
    docs = _docs_of(kind)
    nd, maxlen = oracle.doc_stats(docs)
    r = maxlen + 5 if rate == "above" else rate
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=r) as b:
        b.append_batch(docs)
        b.finish()
        sa = b.suffix_array()
        img = b.sa_file()
        b.save_samples(str(tmp_path / "x"))
        with dsmfm.Searcher(b) as s:
            pos = np.arange(s.n, dtype=np.uint64)
            s.load_samples(img)
            doc, off = s.locate(pos)
            want_doc, want_off = _doc_of(docs, sa)
            assert np.array_equal(doc, want_doc) and np.array_equal(off, want_off)
            s.load_samples(str(tmp_path / "x.sa"))
            doc2, off2 = s.locate(pos)
            assert np.array_equal(doc2, doc) and np.array_equal(off2, off)
            assert s.extract(np.arange(nd)[::-1]) == bytes(docs).split(b"\0")[:-1][::-1]
    if rate == "above":
        assert _sa_sections(img)[0][1] == 0  # no samples at all


def test_pattern_occurrences_in_rank_order(tmp_path):
    """count, then locate_ranges: the brute-force occurrence list of every pattern, in suffix (rank) order."""
    import dsmfm
    docs = oracle.fasta_to_docs(cases.rnd_fasta(61, 400, 80, genome=1200))[0]
    text = bytes(docs)
    rng = np.random.default_rng(61)
    pats = []
    for _ in range(150):
        x = int(rng.integers(0, len(text) - 12))
        p = text[x:x + int(rng.integers(1, 12))].split(b"\0")[0]
        if p:
            pats.append(p)
    pats += [b"ACGTACGTTTTTTTTTTTTAAAA", b"-", b"A", b"C", b"G", b"T", b"N", b"Z"]
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=16) as b:
        b.append_batch(docs)
        b.finish()
        sa = b.suffix_array().astype(np.int64)
        isa = np.empty_like(sa)
        isa[sa] = np.arange(sa.size)
        with dsmfm.Searcher(b) as s:
            s.load_samples(b.sa_file())
            sp, ep = s.count(pats)
            # every pattern's interval followed by an empty one, and one more at the end: they contribute nothing
            sp2 = np.append(np.stack([sp, np.full_like(sp, 9)], axis=1).ravel(), np.uint64(7))
            ep2 = np.append(np.stack([ep, np.full_like(ep, 4)], axis=1).ravel(), np.uint64(6))
            doc, off, starts = s.locate_ranges(sp2, ep2)
            for k, p in enumerate(pats):
                occ, at = [], text.find(p)
                while at >= 0:
                    occ.append(at)
                    at = text.find(p, at + 1)
                occ.sort(key=lambda x: isa[x])
                want_doc, want_off = _doc_of(docs, occ)
                a, z = int(starts[2 * k]), int(starts[2 * k + 1])
                assert np.array_equal(doc[a:z], want_doc) and np.array_equal(off[a:z], want_off), p
                assert starts[2 * k + 2] == starts[2 * k + 1]
            assert int(starts[-1]) == doc.size
            # cap below the total: DSMFM_ELIMIT and the total
            L = dsmfm.lib()
            total = C.c_uint64()
            sp3, ep3 = np.ascontiguousarray(sp2), np.ascontiguousarray(ep2)
            d, o = np.empty(doc.size, dtype=np.uint32), np.empty(doc.size, dtype=np.uint64)
            rc = L.dsmfm_searcher_locate_ranges(s._h, sp3.ctypes.data, ep3.ctypes.data, sp3.size, doc.size - 1, d.ctypes.data,
                                                o.ctypes.data, C.byref(total))
            assert rc == dsmfm.ELIMIT and total.value == doc.size


def test_large_index_locate_on_device_and_extract():
    """25 Mbp sample (C1 shape), rate 124: 4M random positions through locate_device against the suffix array,
    100k random documents through extract."""
    import torch
    import dsmfm
    import dsmgen
    docs = dsmgen.docs(**dsmgen.CONFIGS["C1"])
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA) as b:
        b.append_batch(docs)
        b.finish()
        sa = b.suffix_array()
        with dsmfm.Searcher(b) as s:
            s.load_samples(b.sa_file())
            rng = np.random.default_rng(5)
            m = 4_000_000
            pos = rng.integers(0, s.n, size=m, dtype=np.int64)
            doc = torch.empty(m, dtype=torch.int32, device="cuda")
            off = torch.empty(m, dtype=torch.int64, device="cuda")
            s.locate_device(torch.from_numpy(pos).cuda(), doc, off)
            want_doc, want_off = _doc_of(docs, sa[pos])
            assert np.array_equal(doc.cpu().numpy().view(np.uint32), want_doc)
            assert np.array_equal(off.cpu().numpy().astype(np.uint64), want_off)
            ks = rng.integers(0, dsmgen.CONFIGS["C1"]["n_reads"], size=100_000)
            got = s.extract(ks)
            size = 2 * dsmgen.CONFIGS["C1"]["read_len"] + 2
            for k, g in zip(ks.tolist(), got):
                assert g == docs[k * size:(k + 1) * size - 1].tobytes()


def test_locate_errors(tmp_path):
    """Bad input is refused with DSMFM_EINVAL; nothing is answered from samples that do not fit the index."""
    import dsmfm

    def refused(fn, *a):
        with pytest.raises(dsmfm.DsmfmError) as e:
            fn(*a)
        assert e.value.code == dsmfm.EINVAL, e.value

    img = _golden("reads100.s16.sa")
    with dsmfm.Searcher(os.path.join(GOLDEN, "reads100.fmi")) as s:
        refused(s.locate, [0])
        refused(s.extract, [0])
        refused(s.locate_ranges, [0], [3])
        refused(s.load_samples, os.path.join(GOLDEN, "small_random.s3.sa"))  # another index
        for cut in (0, 10, 23, 24, 1000, 10120, 10150, len(img) // 2, len(img) - 8, len(img) - 1):
            refused(s.load_samples, img[:cut])
        refused(s.load_samples, img + b"\0" * 8)
        tl = bytearray(img)
        at = _sa_sections(img)[2][0] + 16
        tl[at] ^= 1  # textLength[0] +- 1: the lengths no longer add up to n
        refused(s.load_samples, bytes(tl))
        refused(s.locate, [0])  # nothing attached by the refused images
        s.load_samples(img)
        refused(s.locate, [s.n])
        refused(s.locate_ranges, [5], [s.n])
        refused(s.extract, [400])
        doc, off = s.locate([0, s.n - 1])
        assert doc.size == 2
    # same n and document count, other document lengths: the walks of extract do not end where the samples say
    docs_a, docs_b = b"ACG\0TTTAC\0", b"TTTAC\0ACG\0"
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=50) as b:
        b.append_batch(docs_b)
        b.finish()
        img_b = b.sa_file()
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=50) as a:
        a.append_batch(docs_a)
        a.finish()
        with dsmfm.Searcher(a) as s:
            s.load_samples(img_b)
            refused(s.extract, [0])
            s.load_samples(a.sa_file())
            assert s.extract([1, 0]) == [b"TTTAC", b"ACG"]


def test_locate_refuses_walks_longer_than_the_samples_allow():
    """Samples of another index with the same n, document count and (zero) samples pass every check of the image, but
    say the longest document has 4 symbols; this index has one of 7, so walks of up to 7 steps exceed the bound.
    locate and locate_ranges must refuse (DSMFM_EINVAL), not answer; walks within the bound still answer."""
    import torch
    import dsmfm

    def refused(fn, *a):
        with pytest.raises(dsmfm.DsmfmError) as e:
            fn(*a)
        assert e.value.code == dsmfm.EINVAL, e.value

    # in both, document 1's first suffix sorts before document 0's: Doc (document by end-marker rank) agrees
    docs_a, docs_b = b"G\0ACGTTCA\0", b"TTCA\0ACGT\0"
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=50) as b:
        b.append_batch(docs_b)
        b.finish()
        img_b = b.sa_file()
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=50) as a:
        a.append_batch(docs_a)
        a.finish()
        sa = a.suffix_array()
        with dsmfm.Searcher(a) as s:
            s.load_samples(img_b)
            far = int(np.flatnonzero(sa == 9)[0])  # the suffix at offset 7 of document 1: a walk of 7 steps
            near = int(np.flatnonzero(sa == 3)[0])  # offset 1 of document 1: 1 step
            refused(s.locate, [far])
            refused(s.locate, np.arange(s.n))
            refused(s.locate_ranges, [0], [s.n - 1])
            pos = torch.tensor([far], dtype=torch.int64, device="cuda")
            refused(s.locate_device, pos, torch.empty(1, dtype=torch.int32, device="cuda"),
                    torch.empty(1, dtype=torch.int64, device="cuda"))
            doc, off = s.locate([near])
            assert doc.tolist() == [1] and off.tolist() == [1]
            # a position tensor of the wrong type is refused before anything reads it
            with pytest.raises(ValueError):
                s.locate_device(pos.to(torch.int32), torch.empty(1, dtype=torch.int32, device="cuda"),
                                torch.empty(1, dtype=torch.int64, device="cuda"))
