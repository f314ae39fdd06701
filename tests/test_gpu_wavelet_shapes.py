"""GPU suite: the wavelet-tree build (wt_sweep / wt_count / wt_scan / wt_fill, csrc/kernels.cu) and the query kernels
(csrc/search.cu) over every shape of Huffman tree: 0 to 255 internal nodes, shallow and deep (codes of up to 32 bits),
at tile edges and over many tiles, in one piece and assembled from per-slice pieces.

Which kernel builds a tree depends only on its number of internal nodes (= distinct symbols - 1):
  0                       no kernel (the root is a leaf)
  1-8                     wt_sweep_kernel (<4>, <5>, <6> fixed at compile time, <0> otherwise);
                          with DSMFM_WT_SWEEP=0 wt_count / wt_scan / wt_fill, small-table branch
  9-64                    wt_count / wt_fill, node table staged in shared memory
  65-255                  wt_count / wt_fill, node table read from global memory
The expected values come from the oracle (oracle/dsm_oracle.c) and from counting with numpy; the tables under test
never compute them."""
import ctypes as C

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

TILE = 8192               # kWtTile: symbols per CTA of the wavelet-tree kernels
MANY = 33 * TILE + 5      # 34 tiles: the sweep's look-back goes past one window of 32 tiles
BIG = 3_000_017
NEG1 = 2**64 - 1


def _fib(k):
    """F_1 .. F_k = 1, 1, 2, 3, 5, ...: the weights of the deepest Huffman tree over k symbols"""
    f = [1, 1]
    while len(f) < k:
        f.append(f[-1] + f[-2])
    return f[:k]


def _code_bits(counts):
    """Huffman code lengths of the oracle's code table for a 256-entry histogram"""
    tab = (oracle.Code * 256)()
    oracle.lib().dsm_oracle_codetable((C.c_uint64 * 256)(*[int(x) for x in counts]), tab)
    return np.array([tab[c].bits for c in range(256)])


def _max_bits(counts):
    counts = np.asarray(counts)
    return int(_code_bits(counts)[counts > 0].max())


def _alphabet(sigma, rng):
    """sigma distinct byte values with 0 and 255 among them, in shuffled order, so that codes do not follow byte order"""
    if sigma == 1:
        return np.array([rng.choice([0, 255])], dtype=np.uint8)
    rest = rng.permutation(np.arange(1, 255))[: sigma - 2]
    return rng.permutation(np.concatenate([[0, 255], rest])).astype(np.uint8)


def _counts(dist, sigma, n, rng):
    """occurrences of the symbols of rank 0 .. sigma-1, every one >= 1, summing to n"""
    assert n >= sigma
    if dist == "uniform":
        c = np.full(sigma, n // sigma, dtype=np.int64)
        c[: n % sigma] += 1
        return c
    if dist == "skewed":
        w = rng.random(sigma) ** 3 + 1e-3
        return 1 + rng.multinomial(n - sigma, w / w.sum())
    if dist == "dominant":  # one symbol plus singletons
        c = np.ones(sigma, dtype=np.int64)
        c[0] = n - (sigma - 1)
        return c
    assert dist == "fib"
    # the j rarest symbols get F_1 .. F_j -- a chain of j - 1 internal nodes --, the others share the rest equally;
    # of all j, the one that gives the deepest tree with codes of at most 32 bits
    best, best_bits = None, -1
    for j in range(1, sigma + 1):
        f = _fib(j)
        rest = n - sum(f)
        if rest < sigma - j:
            break
        c = np.zeros(sigma, dtype=np.int64)
        c[sigma - j:] = f[::-1]
        if j == sigma:
            c[0] += rest
        else:
            c[: sigma - j] = rest // (sigma - j)
            c[: rest % (sigma - j)] += 1
        bits = _max_bits(np.concatenate([c, np.zeros(256 - sigma, dtype=np.int64)]))
        if best_bits < bits <= 32:
            best, best_bits = c, bits
    return best


def _sequence(sigma, dist, n, seed):
    """A seeded byte sequence of n symbols over sigma distinct bytes.
    late:      the three rarest symbols (counts 1, 1, 2) occur only in the last tile: the nodes that hold only them
               have their first member there
    late_last: the rarest symbol occurs once, at position n - 1"""
    rng = np.random.default_rng(seed)
    alpha = _alphabet(sigma, rng)
    if dist in ("late", "late_last"):
        rare = [1, 1, 2][: min(3, sigma - 1)] if dist == "late" else [1][: sigma - 1]
        base = _counts("uniform", sigma - len(rare), n - sum(rare), rng)
        ranks = np.repeat(np.arange(sigma - len(rare)), base)
        rng.shuffle(ranks)
        seq = np.empty(n, dtype=np.int64)
        if dist == "late":
            lo = min((n - 1) // TILE * TILE, n - sum(rare))
            at = np.sort(rng.choice(np.arange(lo, n), size=sum(rare), replace=False))
        else:
            at = np.array([n - 1][: sum(rare)], dtype=np.int64)
        keep = np.ones(n, dtype=bool)
        keep[at] = False
        seq[keep] = ranks
        seq[at] = rng.permutation(np.repeat(np.arange(sigma - len(rare), sigma), rare))
        return alpha[seq]
    ranks = np.repeat(np.arange(sigma), _counts(dist, sigma, n, rng))
    rng.shuffle(ranks)
    return alpha[ranks]


def _assert_same_fmi(got, want):
    assert oracle.diff_fmi(got, want) == []
    assert got == want


# Every build path x {shallow, deep} x {tile edge, many tiles}; (sigma, distribution, n)
CASES = [
    # no internal node
    (1, "uniform", 1), (1, "uniform", TILE + 1), (1, "uniform", MANY),
    # 1-3 internal nodes: wt_sweep_kernel<0>
    (2, "skewed", 31), (2, "late_last", 32), (3, "dominant", 64), (3, "late", TILE + 2), (4, "fib", 65),
    (4, "uniform", MANY), (4, "late", MANY),
    # 4-6 internal nodes: wt_sweep_kernel<4 / 5 / 6>
    (5, "uniform", 32), (5, "fib", TILE - 1), (6, "skewed", 256), (6, "late", MANY), (7, "fib", MANY),
    (7, "dominant", TILE), (7, "late_last", 257),
    # 7-8 internal nodes: wt_sweep_kernel<0>, nodes 4-7 from the high half of the 8x8 transposes
    (8, "uniform", 33), (8, "fib", TILE + 1), (8, "late", MANY), (8, "skewed", 63), (9, "skewed", 255),
    (9, "fib", MANY), (9, "dominant", 63), (9, "late_last", TILE), (9, "late", MANY), (9, "uniform", BIG),
    # 9-64 internal nodes: node table staged in shared memory
    (10, "uniform", TILE), (10, "fib", MANY), (17, "skewed", 257), (17, "late", MANY), (33, "fib", TILE + 1),
    (33, "dominant", BIG), (64, "uniform", 64), (64, "late_last", TILE - 1), (65, "fib", MANY), (65, "skewed", TILE),
    (65, "late", MANY),
    # 65-255 internal nodes: node table in global memory
    (66, "uniform", 255), (66, "fib", MANY), (66, "late", TILE + 4), (67, "skewed", 256), (67, "late", MANY),
    (128, "skewed", MANY), (128, "dominant", 256), (255, "fib", BIG), (255, "uniform", TILE - 1),
    (256, "late_last", 257), (256, "skewed", BIG), (256, "uniform", MANY), (256, "fib", TILE),
]


def _case_id(case):
    return "s%d-%s-n%d" % case


def _seed(case):
    sigma, dist, n = case
    return sigma * 1_000_003 + n * 7 + sum(dist.encode())


# ---- build against the oracle ------------------------------------------------------------------------------------

# DSMFM_WT_SWEEP=0 only changes the path of trees with at most 8 internal nodes
SWEEP_CASES = [(c, "on") for c in CASES] + [(c, "off") for c in CASES if c[0] <= 9]


@pytest.mark.parametrize("case,sweep", SWEEP_CASES, ids=["%s-sweep_%s" % (_case_id(c), w) for c, w in SWEEP_CASES])
def test_wavelet_tree_matches_oracle(case, sweep, tmp_path, monkeypatch):
    """dsmfm.wavelet_fmi byte for byte against the oracle's HuffWT; then the searcher over the same file against
    counting.  sweep=off: trees of at most 8 internal nodes go through wt_count / wt_scan / wt_fill instead."""
    import dsmfm
    sigma, dist, n = case
    if sweep == "off":
        monkeypatch.setenv("DSMFM_WT_SWEEP", "0")
    seq = _sequence(sigma, dist, n, _seed(case))
    assert seq.size == n and np.unique(seq).size == sigma
    if dist == "fib" and n >= MANY:
        assert _max_bits(np.bincount(seq, minlength=256)) >= min(sigma - 1, 20), "not a deep tree"
    got = dsmfm.wavelet_fmi(seq)
    want = oracle.fmi_from_bwt(seq.tobytes(), 124, 0, 0)
    _assert_same_fmi(got, want)
    if sweep == "on":
        _check_searcher(got, seq, tmp_path, np.random.default_rng(_seed(case)))


def test_sweep_switch_changes_the_kernels_of_a_build(monkeypatch):
    """DSMFM_WT_SWEEP=0 is read at every build: one sweep launch becomes wt_count + wt_scan + wt_fill, same index."""
    import dsmfm
    rng = np.random.default_rng(5)
    docs = b"".join(bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=int(rng.integers(1, 80)))) + b"\0"
                    for _ in range(500))

    def build():
        with dsmfm.Builder(device=0) as b:
            b.append_batch(docs)
            b.finish()
            return b.fmi(), b.stats().kernel_launches

    fmi_on, launches_on = build()
    monkeypatch.setenv("DSMFM_WT_SWEEP", "0")
    fmi_off, launches_off = build()
    monkeypatch.setenv("DSMFM_WT_SWEEP", "1")
    fmi_again, launches_again = build()
    assert launches_off == launches_on + 2 and launches_again == launches_on
    assert fmi_on == fmi_off == fmi_again == oracle.fmi_from_docs(docs)


# ---- the searcher against counting -------------------------------------------------------------------------------

def _positions(n, rng):
    if n <= 2**20:
        return np.arange(n, dtype=np.uint64)
    return np.concatenate([np.arange(4096), np.arange(n - 4096, n),
                           rng.integers(0, n, size=2**20)]).astype(np.uint64)


def _check_searcher(fmi, seq, tmp_path, rng, extra_positions=()):
    """access, rank, lf of the searcher over the .fmi file against counting over seq, and a few hundred random queries
    against the oracle's walk of the same file"""
    import dsmfm
    path = str(tmp_path / "x.fmi")
    with open(path, "wb") as f:
        f.write(fmi)
    n = seq.size
    counts = np.bincount(seq, minlength=256).astype(np.uint64)
    Cc = np.concatenate([np.zeros(1, dtype=np.uint64), np.cumsum(counts, dtype=np.uint64)])
    order = np.argsort(seq, kind="stable")  # positions of every symbol, ascending, symbol after symbol
    own = np.empty(n, dtype=np.uint64)      # occurrences of seq[p] in [0, p]
    own[order] = np.arange(n, dtype=np.uint64) - Cc[seq[order]] + np.uint64(1)
    present = np.flatnonzero(counts)
    absent = sorted({c for c in (0, 255) if not counts[c]} | set(np.flatnonzero(counts == 0)[:3].tolist()))
    with dsmfm.Searcher(path) as s:
        assert s.n == n
        pos = np.concatenate([_positions(n, rng), np.asarray(extra_positions, dtype=np.uint64)])
        sym, rank = s.access(pos)
        assert np.array_equal(sym, seq[pos]), "access: symbol"
        assert np.array_equal(rank, own[pos]), "access: rank"
        # rank / lf of every present symbol (and some absent ones) at sampled positions; positions >= n count as n - 1
        # at every level, also when the root is a leaf; rank(c, -1) = 0
        per = max(4096, 2**20 // len(present))
        q = np.concatenate([pos[:per] if pos.size <= per else rng.choice(pos, size=per, replace=False),
                            np.asarray(extra_positions, dtype=np.uint64),
                            np.array([0, n - 1, n, n + 1, 2 * n + 7, 2**63, NEG1 - 1, NEG1], dtype=np.uint64)]).astype(np.uint64)
        inside = np.minimum(q, np.uint64(n - 1))
        for c in list(present) + absent:
            occ = order[int(Cc[c]):int(Cc[c + 1])]
            want = np.searchsorted(occ, inside, side="right").astype(np.uint64)
            want[q == NEG1] = 0
            assert np.array_equal(s.rank(c, q), want), "rank of byte %d" % c
            want_lf = want + Cc[c] if counts[c] else np.full(q.size, Cc[c], dtype=np.uint64)
            assert np.array_equal(s.lf(c, q), want_lf), "lf of byte %d" % c
        # the oracle's walk of the same file, inside the sequence
        x = oracle.Index(fmi)
        try:
            qi = rng.integers(0, n, size=300).astype(np.uint64)
            qc = np.where(rng.random(300) < 0.9, rng.choice(present, size=300), rng.integers(0, 256, size=300)).astype(np.uint8)
            assert s.rank(qc, qi).tolist() == [x.rank(int(c), int(i)) for c, i in zip(qc, qi)]
            assert s.lf(qc, qi).tolist() == [x.lf(int(c), int(i)) for c, i in zip(qc, qi)]
            sym, rank = s.access(qi)
            assert list(zip(sym.tolist(), rank.tolist())) == [x.access(int(i)) for i in qi]
        finally:
            x.close()


# ---- the 32-bit boundary of the code field ----------------------------------------------------------------------

def _fib_counts(k, rng, terminator=None):
    """histogram of k symbols with weights F_1 .. F_k over shuffled bytes (byte 0 gets weight `terminator` if given)"""
    f = _fib(k)
    vals = rng.permutation(np.arange(1, 256))[:k]
    if terminator is not None:
        vals[f.index(terminator)] = 0
    h = np.zeros(256, dtype=np.int64)
    h[vals] = f
    return h


def test_codes_of_32_bits_build_and_answer_queries(tmp_path):
    """33 symbols with Fibonacci weights (9,227,464 symbols): the two rarest have codes of exactly 32 bits, which the
    .fmi code field holds."""
    import dsmfm
    rng = np.random.default_rng(33)
    h = _fib_counts(33, rng)
    assert _max_bits(h) == 32
    seq = np.repeat(np.arange(256, dtype=np.uint8), h)
    rng.shuffle(seq)
    got = dsmfm.wavelet_fmi(seq)
    _assert_same_fmi(got, oracle.fmi_from_bwt(seq.tobytes(), 124, 0, 0))
    deepest = np.flatnonzero(_code_bits(h) == 32)
    at = np.flatnonzero(np.isin(seq, deepest))
    _check_searcher(got, seq, tmp_path, rng, extra_positions=np.concatenate([at - 1, at, at + 1]).clip(0, seq.size - 1))


def test_builder_with_codes_of_32_bits_locates_and_extracts(tmp_path):
    """The same histogram as 144 documents (the terminator count is one of the weights): the builder's index equals
    the oracle's over the builder's BWT, and locate / extract agree with its suffix array and the documents."""
    import dsmfm
    rng = np.random.default_rng(144)
    h = _fib_counts(33, rng, terminator=144)
    body = np.repeat(np.arange(1, 256, dtype=np.uint8), h[1:])
    rng.shuffle(body)
    cuts = np.sort(rng.choice(np.arange(1, body.size), size=143, replace=False))
    parts = np.split(body, cuts)
    docs = b"".join(p.tobytes() + b"\0" for p in parts)
    nd, maxlen = oracle.doc_stats(docs)
    assert nd == 144 and np.array_equal(np.bincount(np.frombuffer(docs, dtype=np.uint8), minlength=256), h)
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_BWT | dsmfm.FLAG_KEEP_SA) as b:
        b.append_batch(docs)
        b.finish()
        fmi = b.fmi()
        _assert_same_fmi(fmi, oracle.fmi_from_bwt(b.bwt(), 124, nd, maxlen))
        sa = b.suffix_array()
        with dsmfm.Searcher(b) as s:
            s.load_samples(b.sa_file())
            pos = np.concatenate([np.arange(4096), rng.integers(0, s.n, size=200_000)]).astype(np.uint64)
            doc, off = s.locate(pos)
            want_doc, want_off = _doc_of(docs, sa[pos])
            assert np.array_equal(doc, want_doc) and np.array_equal(off, want_off)
            assert s.extract(np.arange(nd)) == [p.tobytes() for p in parts]


def test_codes_of_33_bits_are_refused():
    """34 Fibonacci weights (14,930,351 symbols) need a 33-bit code: the build reports DSMFM_ELIMIT, nothing crashes."""
    import dsmfm
    rng = np.random.default_rng(34)
    h = _fib_counts(34, rng, terminator=144)
    assert _max_bits(h) == 33
    body = np.repeat(np.arange(1, 256, dtype=np.uint8), h[1:])
    rng.shuffle(body)
    cuts = np.sort(rng.choice(np.arange(1, body.size), size=143, replace=False))
    docs = b"".join(p.tobytes() + b"\0" for p in np.split(body, cuts))
    with dsmfm.Builder(device=0) as b:
        b.append_batch(docs)
        with pytest.raises(dsmfm.DsmfmError) as e:
            b.finish()
        assert e.value.code == dsmfm.ELIMIT and "32 bits" in str(e.value)
    with pytest.raises(dsmfm.DsmfmError) as e:
        dsmfm.wavelet_fmi(np.frombuffer(docs, dtype=np.uint8))
    assert "32 bits" in str(e.value)
    # and the library still builds afterwards
    assert dsmfm.build_fmi(b"ACGT\0GAT\0") == oracle.fmi_from_docs(b"ACGT\0GAT\0")


# ---- the wavelet tree assembled from per-slice pieces --------------------------------------------------------------

def _sharded_build(docs, shard_count, span=1):
    """Builds every slice of the global suffix order with its own builder; every slice contributes its bits of every
    wavelet-tree node, the first builder merges them.  Returns (fmi, per-slice byte histograms)."""
    import torch
    import dsmfm
    builders = []
    try:
        for first in range(0, shard_count, span):
            b = dsmfm.Builder(flags=dsmfm.FLAG_KEEP_SA, shard_index=first, shard_count=shard_count,
                              shard_span=min(span, shard_count - first))
            builders.append(b)
            b.append_batch(docs)
            b.build_device()
        hist_all = np.stack([b.slice_hist() for b in builders])
        assert np.array_equal(hist_all.sum(axis=0), np.bincount(np.frombuffer(docs, dtype=np.uint8), minlength=256))
        bufs = []
        for r, b in enumerate(builders):
            bufs.append(torch.empty(b.pieces_bytes(hist_all, r), dtype=torch.uint8, device="cuda"))
            b.build_pieces(hist_all, r, bufs[-1])
        builders[0].assemble_pieces(hist_all, torch.cat(bufs))
        builders[0].fetch()
        return builders[0].fmi(), hist_all
    finally:
        for b in builders:
            b.close()


def _docs_from(body, ndocs, rng, keep_together=()):
    """body cut into ndocs non-empty '\\0'-terminated documents; no cut right behind a position of keep_together"""
    ok = np.ones(body.size, dtype=bool)
    ok[0] = False
    ok[np.asarray(keep_together, dtype=np.int64) + 1] = False
    cuts = np.sort(rng.choice(np.flatnonzero(ok), size=ndocs - 1, replace=False))
    return b"".join(p.tobytes() + b"\0" for p in np.split(body, cuts))


def _piece_docs(kind):
    rng = np.random.default_rng(sum(kind.encode()))
    if kind == "bytes256":  # every byte, uniform: 255 internal nodes
        return _docs_from(rng.integers(1, 256, size=120_000, dtype=np.uint8), 700, rng), None
    if kind == "fib20":  # 20 symbols with Fibonacci weights, the terminator's among them: a chain of 19 nodes
        h = _fib_counts(20, rng, terminator=233)
        body = np.repeat(np.arange(1, 256, dtype=np.uint8), h[1:])
        rng.shuffle(body)
        return _docs_from(body, 233, rng), None
    # "late": bytes 1..250 skewed; 251..253 occur only right before a run of 255s, the largest suffixes, so the BWT
    # holds them only in the last key range
    w = rng.random(250) ** 3 + 1e-3
    body = rng.choice(np.arange(1, 251, dtype=np.uint8), size=90_000, p=w / w.sum())
    at = np.sort(rng.choice(np.arange(10, body.size - 10), size=6, replace=False))
    for k, x in enumerate(at):
        body[x] = 251 + k % 3
        body[x + 1:x + 5] = 255
    return _docs_from(body, 600, rng, keep_together=at), [251, 252, 253]


@pytest.mark.parametrize("shards,span", [(3, 1), (8, 2), (37, 1)])
@pytest.mark.parametrize("kind", ["bytes256", "fib20", "late"])
def test_pieces_of_large_and_deep_trees(kind, shards, span):
    docs, late = _piece_docs(kind)
    fmi, hist_all = _sharded_build(docs, shards, span)
    if late:
        holding = np.flatnonzero(hist_all.sum(axis=1))
        assert set(np.flatnonzero(hist_all[:, late].sum(axis=1)).tolist()) == {int(holding[-1])}
    _assert_same_fmi(fmi, oracle.fmi_from_docs(docs))


# ---- queries on 8-bit indexes --------------------------------------------------------------------------------------

def _doc_of(docs, sa):
    """(document, offset) of text positions `sa` in '\\0'-terminated documents"""
    text = np.frombuffer(bytes(docs), dtype=np.uint8)
    starts = np.concatenate([[0], np.flatnonzero(text == 0)[:-1] + 1]).astype(np.uint64)
    sa = np.asarray(sa, dtype=np.uint64)
    doc = np.searchsorted(starts, sa, side="right") - 1
    return doc.astype(np.uint32), sa - starts[doc]


def _occurrences(text, p):
    """start positions of the overlapping occurrences of p in text (numpy uint8)"""
    m = text.size - len(p) + 1
    if m <= 0:
        return np.zeros(0, dtype=np.int64)
    hit = np.ones(m, dtype=bool)
    for j, c in enumerate(p):
        hit &= text[j:j + m] == c
    return np.flatnonzero(hit)


def _zipf_docs():
    """bytes 1..255 with Zipf-like weights (1 / k^2.5: codes of up to 18 bits) in 3000 documents"""
    rng = np.random.default_rng(255)
    k = np.arange(1, 256)
    w = 1 / k ** 2.5
    cnt = np.maximum(1, np.round(400_000 * w / w.sum())).astype(np.int64)
    body = np.repeat(rng.permutation(np.arange(1, 256)).astype(np.uint8), cnt)
    rng.shuffle(body)
    return _docs_from(body, 3000, rng)


@pytest.mark.parametrize("rate", [1, 7, "above"])
def test_queries_on_an_8_bit_index(rate):
    import dsmfm
    docs = _zipf_docs()
    text = np.frombuffer(docs, dtype=np.uint8)
    nd, maxlen = oracle.doc_stats(docs)
    assert _max_bits(np.bincount(text, minlength=256)) >= 17
    r = maxlen + 3 if rate == "above" else rate
    rng = np.random.default_rng(7)
    pats = []
    for _ in range(300):
        x = int(rng.integers(0, text.size - 8))
        p = bytes(text[x:x + int(rng.integers(1, 8))]).split(b"\0")[0]
        if p:
            pats.append(p)
    pats += [bytes([c]) for c in range(1, 256)]
    pats += [bytes(rng.integers(1, 256, size=4, dtype=np.uint8)) for _ in range(20)]  # almost surely absent
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=r) as b:
        b.append_batch(docs)
        b.finish()
        sa = b.suffix_array().astype(np.int64)
        isa = np.empty_like(sa)
        isa[sa] = np.arange(sa.size)
        with dsmfm.Searcher(b) as s:
            s.load_samples(b.sa_file())
            sp, ep = s.count(pats)
            occ = [_occurrences(text, p) for p in pats]
            got = np.where(sp <= ep, ep - sp + np.uint64(1), np.uint64(0))
            assert got.tolist() == [o.size for o in occ]
            # every byte to the left of every pattern at once: occurrences of c + pattern = occurrences of the pattern
            # behind a c (byte 0 is left out: in front of the first document the index wraps round to the last one)
            so, eo = s.extend(sp, ep, bytes(range(256)))
            n_left = np.where(so <= eo, eo - so + np.uint64(1), np.uint64(0))
            for j, o in enumerate(occ):
                want = np.bincount(text[o[o > 0] - 1], minlength=256)
                assert np.array_equal(n_left[j, 1:], want[1:]), pats[j]
            for j in rng.choice(len(pats), size=40, replace=False):
                lsp, lep = s.count([bytes([c]) + pats[j] for c in range(256)])
                full = sp[j] <= ep[j]
                assert np.array_equal(so[j], lsp if full else np.full(256, sp[j])), pats[j]
                assert np.array_equal(eo[j], lep if full else np.full(256, ep[j])), pats[j]
            # locate_ranges: the occurrences of every pattern in suffix order
            doc, off, starts = s.locate_ranges(sp, ep)
            for j, o in enumerate(occ):
                o = o[np.argsort(isa[o])]
                want_doc, want_off = _doc_of(docs, o)
                a, z = int(starts[j]), int(starts[j + 1])
                assert np.array_equal(doc[a:z], want_doc) and np.array_equal(off[a:z], want_off), pats[j]
            doc, off = s.locate(np.arange(s.n, dtype=np.uint64))
            want_doc, want_off = _doc_of(docs, sa)
            assert np.array_equal(doc, want_doc) and np.array_equal(off, want_off)
            assert s.extract(np.arange(nd)[::-1]) == docs.split(b"\0")[:-1][::-1]
