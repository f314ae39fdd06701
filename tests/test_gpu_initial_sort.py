"""GPU suite: the initial suffix sort of an unsharded build, stage by stage (dsmfm.initial_sort stops after the group
heads): the first keys and their digit counts, the one-sweep passes across tiles and portions, the group heads, the
difference bits, `remaining` and the carried BWT, each against a numpy reference restated from the raw bytes
(DESIGN.md section 3, items 2-4).  Also: keying in word ranges (a batch streaming in from the host), and streamed
batches whose speculative pack is kept."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

CHUNK = 1 << 24
PIECE = 21 * 3145728  # bytes per piece of a batch that streams in from the host (append_pipelined)


def shape(docs, first_key_bits=0):
    """(code map, bits, first_syms, key_bits, carry) of an unsharded build of these documents."""
    present = np.bincount(docs, minlength=256) > 0
    present[0] = False
    code = np.zeros(256, np.uint8)
    sigma = int(present.sum())
    code[present] = np.arange(1, sigma + 1, dtype=np.uint8)
    bits = 3 if sigma <= 7 else (4 if sigma <= 15 else 8)
    spw = 64 // bits
    fkb = 48 if first_key_bits <= 0 else first_key_bits
    if fkb < 8 or fkb > spw * bits:
        fkb = spw * bits
    fs = max(1, fkb // bits)
    return code, bits, fs, fs * bits, fs * bits + bits <= 64


def keys_of(codes, lo, hi, bits, fs, key_bits, carry):
    """Keys of suffixes [lo, hi): the next fs codes, zero from the first terminator on, most significant first;
    with carry the code of the symbol before the suffix (0 at position 0) just above them.  `codes` has at least
    fs zeros behind the text."""
    k = np.zeros(hi - lo, np.uint64)
    alive = np.ones(hi - lo, bool)
    for j in range(fs):
        c = codes[lo + j:hi + j]
        k |= np.where(alive, c, 0).astype(np.uint64) << np.uint64(bits * (fs - 1 - j))
        alive &= c != 0
    if carry:
        prev = codes[lo - 1:hi - 1] if lo else np.concatenate([[0], codes[:hi - 1]]).astype(np.uint8)
        k |= prev.astype(np.uint64) << np.uint64(key_bits)
    return k


def _pack_bits(flags, fill):
    """bool flags -> u32 words, bit i of word i // 32 = flags[i]; positions behind the flags take `fill`."""
    pad = (-flags.size) % 32
    if pad:
        flags = np.concatenate([flags, np.full(pad, fill)])
    return np.packbits(flags, bitorder="little").view("<u4")


def check(docs, out, first_key_bits=0):
    """Asserts that every product of dsmfm.initial_sort(docs, first_key_bits) equals the reference."""
    n = docs.size
    code, bits, fs, key_bits, carry = shape(docs, first_key_bits)
    assert (out["bits"], out["first_syms"], out["carry"]) == (bits, fs, int(carry))
    kmask = np.uint64((1 << key_bits) - 1)
    field = np.uint64((1 << bits) - 1)
    codes = np.zeros(n + fs + 1, np.uint8)
    codes[:n] = code[docs]
    keys, sk, sa = out["keys"], out["sorted_keys"], out["sa"]
    # keys and their digit counts
    npass = (key_bits + 7) // 8
    hist = np.zeros((8, 256), np.uint64)
    for lo in range(0, n, CHUNK):
        hi = min(n, lo + CHUNK)
        want = keys_of(codes, lo, hi, bits, fs, key_bits, carry)
        bad = np.flatnonzero(keys[lo:hi] != want)
        assert bad.size == 0, "key of suffix %d: %#x, want %#x" % (lo + bad[0], keys[lo + bad[0]], want[bad[0]])
        m = want & kmask
        for q in range(npass):
            hist[q] += np.bincount(((m >> np.uint64(8 * q)) & np.uint64(255)).astype(np.intp), minlength=256).astype(np.uint64)
    for q in range(8):
        assert np.array_equal(out["hist"][q], hist[q]), "digit counts of pass %d" % q
    # the sort: a permutation, ordered under the mask, stable, carrying its keys
    mark = np.zeros(n, bool)
    mark[sa] = True
    assert mark.all(), "sa is not a permutation"
    del mark
    if n <= CHUNK:
        assert np.array_equal(sa, np.argsort(keys & kmask, kind="stable").astype(np.uint32))
    remaining = 0
    for lo in range(0, n, CHUNK):
        hi = min(n, lo + CHUNK)
        s = sa[lo:hi]
        k = sk[lo:hi]
        assert np.array_equal(k, keys[s]), "sorted keys are not the keys of their positions"
        m = k & kmask
        prev = sk[lo - 1:hi - 1] if lo else np.concatenate([[sk[0] ^ kmask], sk[:hi - 1]]).astype(np.uint64)
        pm = prev & kmask
        assert (m >= pm)[1 if lo == 0 else 0:].all(), "not sorted"
        tie = m == pm
        if lo == 0:
            tie[0] = False
        ps = sa[lo - 1:hi - 1] if lo else np.concatenate([[0], sa[:hi - 1]]).astype(np.uint32)
        assert (s[tie] > ps[tie]).all(), "not stable"
        # heads, difference bits, remaining
        head = (m != pm) | ((m & field) == 0)
        if lo == 0:
            head[0] = True
        w0, w1 = lo // 32, (hi + 31) // 32
        assert np.array_equal(out["head"][w0:w1], _pack_bits(head, True)), "head bits in words %d..%d" % (w0, w1)
        if carry:
            dif = ~head & (((k >> np.uint64(key_bits)) & field) != ((prev >> np.uint64(key_bits)) & field))
            assert np.array_equal(out["diff"][w0:w1], _pack_bits(dif, False)), "difference bits in words %d..%d" % (w0, w1)
            bw = np.where(s > 0, docs[np.maximum(s.astype(np.int64) - 1, 0)], 0).astype(np.uint8)
            assert np.array_equal(out["bwt"][lo:hi], bw), "carried BWT"
        nxt_head = np.empty_like(head)
        nxt_head[:-1] = head[1:]
        if hi < n:
            a, b = sk[hi - 1] & kmask, sk[hi] & kmask
            nxt_head[-1] = a != b or (b & field) == 0
        else:
            nxt_head[-1] = True
        remaining += int((~(head & nxt_head)).sum())
    if not carry:  # nothing carried: diff and bwt left as the caller had them (zero)
        assert not out["diff"].any() and not out["bwt"].any()
    assert out["remaining"] == remaining


# ---- inputs ---------------------------------------------------------------------------------------------------

def alphabet(size, seed):
    """`size` distinct non-zero byte values in shuffled order, 1 and 255 among them."""
    rng = np.random.default_rng(seed)
    rest = rng.choice(np.arange(2, 255, dtype=np.uint8), size - 2, replace=False)
    return rng.permutation(np.concatenate([[1, 255], rest]).astype(np.uint8))


def random_docs(n, alpha, seed, minlen=1, maxlen=60):
    """Exactly n bytes of non-empty documents over `alpha`, every symbol of it present when n allows."""
    rng = np.random.default_rng(seed)
    out = rng.choice(alpha, size=n).astype(np.uint8)
    k = min(alpha.size, n - 1)
    out[:k] = alpha[:k]
    lens = rng.integers(minlen, maxlen + 1, size=n // max(1, minlen) + 2)
    ends = np.cumsum(lens + 1) - 1
    out[ends[ends <= n - 3]] = 0
    out[n - 1] = 0
    return out


def docs_of(lengths, alpha, seed):
    """Documents of the given lengths (terminator not counted), symbols drawn from alpha."""
    rng = np.random.default_rng(seed)
    parts = [np.append(rng.choice(alpha, size=L).astype(np.uint8), np.uint8(0)) for L in lengths]
    return np.concatenate(parts)


def run(docs, first_key_bits=0, word_cuts=None):
    import dsmfm
    out = dsmfm.initial_sort(docs, first_key_bits=first_key_bits, word_cuts=word_cuts)
    check(docs, out, first_key_bits)
    return out


ALPHABETS = [5, 7, 8, 15, 16, 255]  # 3-bit (reads, largest), 4-bit (smallest, largest), 8-bit (smallest, largest)
# +-1 around multiples of 21 / 16 / 8 symbols (a packed word), the heads chunk (32 * U ranks, U = 4 and 8), the key
# tile (128 words: 1024, 2048 and 2688 symbols) and the sweep tile (4096 pairs); 3 M spans many tiles of each
SIZES = [2, 3, 7, 8, 9, 15, 16, 17, 20, 21, 22, 41, 43, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024,
         1025, 2047, 2048, 2049, 2687, 2688, 2689, 4095, 4096, 4097, 8191, 8193, 3_000_017]


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("sigma", ALPHABETS)
def test_initial_sort_matches_the_reference(sigma, n):
    run(random_docs(n, alphabet(sigma, sigma), seed=n * 7 + sigma))


FIRST_KEY_BITS = [0, 54, 56, 63, 64, 9, 24]  # default (48), long first keys, whole word (no carry), short keys


def _shaped_docs(kind, sigma, fs):
    a = alphabet(sigma, 100 + sigma)
    spw = 64 // (3 if sigma <= 7 else (4 if sigma <= 15 else 8))
    if kind == "one_symbol":
        return docs_of([1] * 3000, a, 1)
    if kind == "around_first_key":  # terminator in the last field of the key, just past it, one field short
        short = max(1, fs - 1)  # (documents are never empty)
        return docs_of([short, fs, fs + 1] * 700 + [fs + 1, fs, short] * 300, a[:2], 2)
    if kind == "poly_a":  # one giant tie group, then many equal documents of it
        return np.concatenate([np.full(9000, a[0], np.uint8), [0], np.tile(np.append(np.full(40, a[0], np.uint8), 0), 200)])
    if kind == "duplicates":
        d = docs_of([37, 5, 80], a, 3)
        return np.tile(d, 150)
    if kind == "word_end_terminators":  # every terminator is the last symbol of a packed word
        return docs_of([spw - 1] * 600 + [2 * spw - 1] * 300, a, 4)
    raise ValueError(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("first_key_bits", FIRST_KEY_BITS)
@pytest.mark.parametrize("kind", ["one_symbol", "around_first_key", "poly_a", "duplicates", "word_end_terminators"])
@pytest.mark.parametrize("sigma", [5, 8, 255])
def test_initial_sort_document_shapes(sigma, kind, first_key_bits):
    fs = shape(np.append(alphabet(sigma, 100 + sigma), np.uint8(0)), first_key_bits)[2]
    run(_shaped_docs(kind, sigma, fs), first_key_bits)


def _cut_sets(words, seed):
    rng = np.random.default_rng(seed)
    rnd = np.unique(rng.integers(1, words, size=min(40, words - 1)))
    return {"random": rnd, "127": [127], "128": [128], "129": [129], "127_128_129": [127, 128, 129]}


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [5, 15, 255])
def test_keying_in_word_ranges_equals_the_uncut_call(sigma):
    """A batch streaming in from the host is packed and keyed word range by word range; every cut gives the products
    of the uncut call (which is checked against the reference), on 3-, 4- and 8-bit alphabets."""
    docs = random_docs(3_000_017, alphabet(sigma, sigma), seed=sigma)
    whole = run(docs)
    words = -(-docs.size // (64 // whole["bits"]))
    cases = _cut_sets(words, sigma)
    small = random_docs(5000, alphabet(sigma, sigma), seed=sigma + 1)
    small_words = -(-small.size // (64 // whole["bits"]))
    for name, cuts in list(cases.items()) + [("every_word", None)]:
        d, c = (small, np.arange(1, small_words)) if cuts is None else (docs, cuts)
        got = run(d, word_cuts=c)
        want = whole if cuts is not None else run(d)
        for key in ("keys", "hist", "sorted_keys", "sa", "head", "diff", "bwt"):
            assert np.array_equal(got[key], want[key]), "cuts %s: %s differ" % (name, key)
        assert got["remaining"] == want["remaining"]


# ---- the entry point refuses malformed input before it launches anything (no GPU needed) ----------------------

def _raw_call(docs, n=None, cuts=(), first_key_bits=0):
    import dsmfm
    L = dsmfm.lib()
    n = docs.size if n is None else n
    m = max(1, docs.size)
    bufs = [np.zeros(m, np.uint64), np.zeros(2048, np.uint64), np.zeros(m, np.uint64), np.zeros(m, np.uint32),
            np.zeros(m, np.uint32), np.zeros(m, np.uint32), np.zeros(m, np.uint8), np.zeros(1, np.uint64)]
    c = np.ascontiguousarray(cuts, dtype=np.uint64)
    ints = [C.c_int() for _ in range(3)]
    return L.dsmfm_dbg_initial_sort(0, docs.ctypes.data if docs.size else None, n, first_key_bits,
                                    c.ctypes.data if c.size else None, c.size, *[b.ctypes.data for b in bufs],
                                    *[C.byref(i) for i in ints])


@pytest.mark.parametrize("case", ["empty", "unterminated", "empty_first_doc", "empty_doc_inside", "too_long",
                                  "cut_zero", "cut_past_text", "cuts_not_increasing", "cuts_equal"])
def test_initial_sort_refuses_malformed_input(case):
    import dsmfm
    ok = np.frombuffer(b"ACGT\0GATTACA\0" * 20, np.uint8).copy()  # 260 symbols: 13 words of 21 3-bit symbols
    args = {"empty": (np.zeros(0, np.uint8),), "unterminated": (ok[:-1],),
            "empty_first_doc": (np.concatenate([[0], ok]).astype(np.uint8),),
            "empty_doc_inside": (np.concatenate([ok[:5], [0], ok[5:]]).astype(np.uint8),),
            "too_long": (ok, (1 << 32) - 2112), "cut_zero": (ok, None, [0, 3]), "cut_past_text": (ok, None, [3, 13]),
            "cuts_not_increasing": (ok, None, [5, 3]), "cuts_equal": (ok, None, [3, 3])}[case]
    assert _raw_call(*args) == dsmfm.EINVAL


# ---- across portions: a pass runs as one launch per 2^29 pairs --------------------------------------------------

PORTION = 1 << 29


def _dna_keys(i):
    """48-bit keys of 16 three-bit fields with codes 4..7 (few digit values), from a hash of the index i; every
    fifth block of 2^20 indices holds one key (long equal runs, across portion boundaries too)."""
    i = i.astype(np.uint64)
    h = (i + np.uint64(0x9E3779B97F4A7C15)) * np.uint64(0xBF58476D1CE4E5B9)
    h ^= h >> np.uint64(31)
    h *= np.uint64(0x94D049BB133111EB)
    h ^= h >> np.uint64(29)
    k = (h & np.uint64(0x6DB6DB6DB6DB)) | np.uint64(0x924924924924)  # every 3-bit field 0b1xx
    run = ((i >> np.uint64(20)) % np.uint64(5)) == 0
    k[run] = np.uint64(0xB6DB6DB6DB6D)
    return k


@pytest.mark.gpu
@pytest.mark.parametrize("n", [PORTION + 4097, 2 * PORTION])
def test_radix_sort_across_portions(n):
    """dsmfm.radix_sort over more than one portion, checked in O(n): sorted, stable, a permutation, and every key
    the key of its position.  Host memory: 12 bytes per pair plus chunk temporaries, about 14 GB at 2^30 pairs."""
    import dsmfm
    if os.environ.get("DSMFM_TEST_SMALL"):
        pytest.skip("needs more than 2^29 pairs")
    keys = np.empty(n, np.uint64)
    for lo in range(0, n, CHUNK):
        keys[lo:lo + CHUNK] = _dna_keys(np.arange(lo, min(n, lo + CHUNK)))
    vals = np.arange(n, dtype=np.uint32)
    dsmfm.radix_sort(keys, vals, 0, 48)
    mark = np.zeros(n, bool)
    mark[vals] = True
    assert mark.all(), "not a permutation"
    del mark
    for lo in range(0, n, CHUNK):
        hi = min(n, lo + CHUNK)
        a = lo - 1 if lo else 0
        k, v = keys[a:hi], vals[a:hi]
        assert np.array_equal(keys[lo:hi], _dna_keys(vals[lo:hi])), "keys near %d are not the keys of their positions" % lo
        assert (k[1:] >= k[:-1]).all(), "not sorted near %d" % lo
        tie = k[1:] == k[:-1]
        assert (v[1:][tie] > v[:-1][tie]).all(), "not stable near %d" % lo


@pytest.mark.gpu
def test_initial_sort_across_portions():
    """About 600 M symbols of C3-shaped reads (more than one 2^29-pair portion per pass) against the reference in
    O(n).  Host memory: about 25 bytes per symbol, 15 GB."""
    import dsmgen
    if os.environ.get("DSMFM_TEST_SMALL"):
        pytest.skip("needs more than 2^29 suffixes")
    kw = dict(dsmgen.CONFIGS["C3"], n_reads=2_970_000)
    docs = dsmgen.docs(**kw)
    assert docs.size > PORTION
    run(docs)


# ---- batches that stream in from pinned host memory and keep their speculative pack ----------------------------

def _streamed_cases(name):
    if name == "4bit":
        return random_docs(3 * PIECE + 1_000_003, alphabet(12, 41), seed=41, minlen=40, maxlen=160)
    if name == "8bit":
        return random_docs(3 * PIECE + 2_000_001, alphabet(200, 42), seed=42, minlen=40, maxlen=160)
    if name == "exact_three_pieces":
        return random_docs(3 * PIECE, np.frombuffer(b"ACGTN", np.uint8), seed=43, minlen=90, maxlen=110)
    if name == "last_piece_one_short_doc":
        d = random_docs(3 * PIECE, np.frombuffer(b"ACGT", np.uint8), seed=44, minlen=90, maxlen=110)
        return np.concatenate([d, np.frombuffer(b"GA\0", np.uint8)])
    raise ValueError(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4bit", "8bit", "exact_three_pieces", "last_piece_one_short_doc"])
def test_streamed_batch_keeps_its_speculation(name):
    """A host batch of at least three 63 MiB pieces is packed and keyed piece by piece behind the copy, with the
    alphabet of its first piece; here the guess holds, the work is kept (stats.streamed), and the index equals that
    of the same documents appended from device memory."""
    import torch
    import dsmfm
    docs = _streamed_cases(name)
    host = torch.from_numpy(docs).pin_memory()
    with dsmfm.Builder() as b:
        b.append_batch(host)
        b.finish()
        assert b.stats().streamed == 1
        got = hashlib.sha256(b.fmi()).hexdigest()
    with dsmfm.Builder() as b:
        b.append_batch_device(host.cuda())
        b.finish()
        assert b.stats().streamed == 0
        want = hashlib.sha256(b.fmi()).hexdigest()
    assert got == want
