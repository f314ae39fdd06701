"""GPU suite: the suffix-order refinement on its own (DESIGN.md section 3, item 5), through dsmfm.refine -- the
build's own driver run on a state the test lays out: tie groups of chosen sizes at chosen slots, at a chosen depth.
Every result is checked against the C oracle's suffix order: each input group's members sorted by their rank in
the full suffix array (or, for the case too large for the oracle, by their bytes from `depth` up to and including
the terminator, ties by position).  Every case also asserts that it reached the path it is named for (the `paths`
bits and the counters of dsmfm_stats), so a case that stops reaching its edge fails instead of passing quietly."""
import os
import zlib

import numpy as np
import pytest

KW = 1024          # kRefWindow: slots whose group heads one CTA owns
GROUP_MAX = 768    # kRwGroupMax: larger groups (or a last group reaching further) take the large-group path
TILE = 8192        # slots of one compaction tile (kActTileWords head words)


# ---- texts and layouts ----------------------------------------------------------------------------------------

def alphabet(size, seed):
    """`size` distinct non-zero byte values in shuffled order, 1 and 255 among them."""
    rng = np.random.default_rng(seed)
    rest = rng.choice(np.arange(2, 255, dtype=np.uint8), size - 2, replace=False)
    return rng.permutation(np.concatenate([[1, 255], rest]).astype(np.uint8))


class Text:
    """Documents appended one by one; family() returns the positions of suffixes that share a given core."""

    def __init__(self, sigma=5, seed=0):
        self.alpha = alphabet(sigma, sigma)
        self.rng = np.random.default_rng(seed)
        self.parts, self.n = [], 0
        self.doc(self.alpha)  # every symbol occurs: the alphabet fixes the bits per symbol

    def doc(self, body):
        p = self.n
        self.parts.append(np.append(np.asarray(body, np.uint8), np.uint8(0)))
        self.n += len(body) + 1
        return p

    def random(self, lo, hi, alpha=None):
        return self.rng.choice(self.alpha if alpha is None else alpha, size=int(self.rng.integers(lo, hi + 1)))

    def filler(self, nsyms, lo=20, hi=120):
        """Random documents of about nsyms symbols (their suffixes fill the singleton slots)."""
        end = self.n + nsyms
        while self.n < end:
            self.doc(self.random(lo, hi))

    def family(self, k, core, tails=None, x=None):
        """k documents x_i + core + tail_i: the positions of `core` in them, members that share len(core) symbols.
        x: one symbol for all (a group with a single BWT symbol), a sequence of them, or None: random per document,
        the second one differing from the first (mixed).  tails: a function i -> tail, by default 0..40 symbols
        over two letters (long ties, terminators at every offset)."""
        core = np.asarray(core, np.uint8)
        two = self.alpha[:2]
        if x is None:
            x = self.rng.choice(self.alpha, size=k)
            if k >= 2 and x[1] == x[0]:
                x[1] = self.alpha[(int(np.flatnonzero(self.alpha == x[0])[0]) + 1) % self.alpha.size]
        pos = []
        for i in range(k):
            xi = x[i] if np.ndim(x) else x
            tail = tails(i) if tails is not None else self.random(0, 40, two)
            pos.append(self.doc(np.concatenate([[xi], core, tail]).astype(np.uint8)) + 1)
        return np.array(pos, np.int64)

    def core(self, length):
        return self.rng.choice(self.alpha, size=length).astype(np.uint8)

    def docs(self):
        return np.concatenate(self.parts)


def layout(n, m, placed):
    """(sa, head words) of m slots: each (slot, members) of `placed` is one group, every other slot a singleton
    holding a position no group uses.  Members are put in ascending order, as a stable initial sort leaves them."""
    sa = np.full(m, -1, np.int64)
    head = np.ones(m, bool)
    used = np.zeros(n, bool)
    for slot, mem in placed:
        mem = np.sort(np.asarray(mem, np.int64))
        assert slot + mem.size <= m and (sa[slot:slot + mem.size] < 0).all(), "groups overlap"
        sa[slot:slot + mem.size] = mem
        head[slot + 1:slot + mem.size] = False
        used[mem] = True
    free = np.flatnonzero(sa < 0)
    fill = np.flatnonzero(~used)
    assert fill.size >= free.size, "text too short for the fillers"
    sa[free] = fill[:free.size]
    return sa.astype(np.uint64), pack_bits(head)


def pack_bits(flags):
    pad = (-flags.size) % 32
    return np.packbits(np.concatenate([flags, np.ones(pad, bool)]), bitorder="little").view("<u4").copy()


def head_flags(head, m):
    return np.unpackbits(head.view(np.uint8), bitorder="little")[:m].astype(bool)


# ---- references -----------------------------------------------------------------------------------------------

def oracle_rank(docs):
    import oracle
    _, sa = oracle.bwt(docs.tobytes(), want_sa=True)
    rank = np.empty(docs.size, np.int64)
    rank[sa.astype(np.int64)] = np.arange(docs.size)
    return rank


def bwt_of(docs, sa):
    s = sa.astype(np.int64)
    return np.where(s > 0, docs[np.maximum(s - 1, 0)], 0).astype(np.uint8)


def group_ref(docs, sa, hf, depth):
    """Each group of >= 2 members sorted by its bytes from `depth` up to and including the terminator, ties by
    position (for inputs too large for the oracle)."""
    want = sa.astype(np.int64).copy()
    term = np.flatnonzero(docs == 0)
    starts = np.flatnonzero(hf)
    ends = np.append(starts[1:], hf.size)
    for g in np.flatnonzero(ends - starts >= 2):
        mem = want[starts[g]:ends[g]]
        t = term[np.searchsorted(term, mem)]
        keyed = sorted((docs[p + depth:e + 1].tobytes(), p) for p, e in zip(mem, t))
        want[starts[g]:ends[g]] = [p for _, p in keyed]
    return want


def first_round_big(hf):
    """Members of the groups the first launch leaves to the large-group path: a window's last group when it reaches
    more than 768 slots behind its head (kernels.cu, ownership of the CTA); every slot from m on is a head."""
    m = hf.size
    heads = np.append(np.flatnonzero(hf), m)
    total = 0
    for w in range(m // KW):  # (a window that reaches past m ends in head bits)
        i = int(np.searchsorted(heads, (w + 1) * KW)) - 1
        if i >= 0 and heads[i] >= w * KW and heads[i + 1] - heads[i] > GROUP_MAX:
            total += int(heads[i + 1] - heads[i])
    return total


def run(docs, sa, head, depth, keep_sa=False, lo_bits=0, rank=None, compact_off=False):
    """dsmfm.refine on the state, every product checked; returns its result."""
    import dsmfm
    m = sa.size
    out = dsmfm.refine(docs, sa, head, depth, keep_sa=keep_sa, lo_bits=lo_bits)
    hf = head_flags(head, m)
    gid = np.cumsum(hf) - 1
    s_in = sa.astype(np.int64)
    if rank is None and docs.size <= 1 << 22:
        rank = oracle_rank(docs)
    want = s_in[np.lexsort((rank[s_in], gid))] if rank is not None else group_ref(docs, sa, hf, depth)
    got = out["sa"].astype(np.int64)
    size = np.bincount(gid)
    in_group = size[gid] >= 2
    # 1. every group's slots hold a permutation of its members
    assert np.array_equal(got[~in_group], s_in[~in_group]), "a singleton moved"
    ig = np.flatnonzero(in_group)
    g, a, b = gid[ig], got[ig], s_in[ig]
    assert np.array_equal(a[np.lexsort((a, g))], b[np.lexsort((b, g))]), "a group lost or gained members"
    # 2. the BWT at every slot
    wbwt = bwt_of(docs, want)
    bad = np.flatnonzero(out["bwt"] != wbwt)
    assert bad.size == 0, "BWT differs at %d slots, first %d (group %d)" % (bad.size, bad[0], gid[bad[0]])
    if not out["paths"] & dsmfm.RPATH_COMPACT:  # (the dense copies send only their BWT bytes back)
        assert np.array_equal(out["bwt"], bwt_of(docs, got)), "BWT bytes do not travel with their suffixes"
    # 3. the full order
    if keep_sa:
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, "suffix order differs at %d slots, first %d" % (bad.size, bad[0])
    # 4. what was counted
    st = out["stats"]
    remaining = int(ig.size)
    b_in = bwt_of(docs, b).astype(np.int64)
    gmin = np.full(size.size, 256)
    gmax = np.full(size.size, -1)
    np.minimum.at(gmin, g, b_in)
    np.maximum.at(gmax, g, b_in)
    mixed_slot = gmin[g] != gmax[g]
    mixed = int(mixed_slot.sum())
    if keep_sa or compact_off:
        assert st["refine_members"] == remaining
        assert st["active"][0] == remaining
    else:
        assert st["refine_members"] == mixed
        assert st["active"][0] == (remaining if mixed else 0)
        assert bool(out["paths"] & dsmfm.RPATH_COMPACT) == (mixed > 0 and 2 * mixed <= remaining)
        if not mixed:  # nothing to sort: the state comes back as it went in
            assert np.array_equal(got, s_in) and st["rounds"] == 0
    assert st["rounds"] == st["refine_launches"]
    if st["refine_launches"]:
        assert bool(out["paths"] & dsmfm.RPATH_ORDER) == keep_sa
        assert bool(out["paths"] & dsmfm.RPATH_WIDE) == (lo_bits > 0)
        sigma = int((np.bincount(docs, minlength=256)[1:] > 0).sum())
        assert (out["paths"] >> dsmfm.RPATH_BITS_SHIFT) & 15 == (3 if sigma <= 7 else (4 if sigma <= 15 else 8))
    # the large-group path takes at least the groups that the first launch cannot own
    big1 = first_round_big(hf[ig[mixed_slot]] if out["paths"] & dsmfm.RPATH_COMPACT else hf)
    assert st["fallback_elems"] >= big1
    out.update(remaining=remaining, mixed=mixed, big1=big1)
    return out


MODES = ["keep_sa", "bwt_compact", "bwt_in_place"]  # full order; BWT order on dense copies; BWT order in place


def state(t, m, placed, mode):
    """(docs, sa, head) of m slots laid out as `placed` (every group mixed).  In mode bwt_compact the same slots
    become the dense copy: each run of singleton slots between the groups is taken by mixed groups of two or three
    members, and around them lie groups with a single BWT symbol holding 2 m members (5 in front, so that the dense
    index of a warp's first slot is not a multiple of 32).  The compaction then keeps exactly slots [0, m), in
    place, and carves its scratch and dense arrays out of the key buffers of the range."""
    if mode != "bwt_compact":
        t.filler(m)
        docs = t.docs()
        return (docs,) + layout(docs.size, m, placed)
    used = np.zeros(m + 1, bool)
    used[m] = True
    for slot, mem in placed:
        used[slot:slot + len(mem)] = True
    core = t.core(20)
    a0, a1 = t.alpha[0], t.alpha[1]
    front = 5
    dense = list(placed)
    slot = 0
    while slot < m:
        if used[slot]:
            slot += 1
            continue
        run_len = int(np.argmax(used[slot:]))
        assert run_len >= 2, "a single free slot at %d cannot hold a mixed group" % slot
        for k in [2] * (run_len // 2 - 1) + [2 + run_len % 2]:
            dense.append((slot, t.family(k, core, x=[a0, a1, a0][:k])))
            slot += k
    real = [(front + s, mem) for s, mem in dense] + [(0, t.family(front, core, x=a1))]
    for slot in range(front + m, 3 * m, 50):
        real.append((slot, t.family(min(50, 3 * m - slot), core, x=a1)))
    docs = t.docs()
    return (docs,) + layout(docs.size, 3 * m, real)


def run_mode(mode, monkeypatch, docs, sa, head, depth, **kw):
    import dsmfm
    if mode == "bwt_in_place":
        monkeypatch.setenv("DSMFM_REFINE_COMPACT", "0")
    out = run(docs, sa, head, depth, keep_sa=mode == "keep_sa", compact_off=mode == "bwt_in_place", **kw)
    if mode == "bwt_compact":  # dense copies carved out of the key buffers (see state())
        assert out["paths"] & (dsmfm.RPATH_COMPACT | dsmfm.RPATH_SCRATCH_ALLOC | dsmfm.RPATH_DENSE_ALLOC) == \
            dsmfm.RPATH_COMPACT
    else:
        assert not out["paths"] & dsmfm.RPATH_COMPACT
    return out


# ---- group size against the ranking paths -----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("size", [2, 31, 32, 33, 63, 64, 65, 1000])
def test_group_size(size, mode, monkeypatch):
    """Groups of `size` members at depth 16 (a shared core, tails over two letters): one at lane 0 of a warp-load,
    one continuing past lane 31, and a single group of 1000 members inside one window, which its CTA refines (only a
    window's last group can be too large for it)."""
    t = Text(5, size)
    core = t.core(16)
    fams = [t.family(size, core) for _ in range(2)]
    second = (64 + size + 32) // 32 * 32 + 31  # at lane 31: it continues into the next head word
    placed = [(64, fams[0]), (second, fams[1])] if size < 900 else [(10, fams[0])]
    docs, sa, head = state(t, 2 * KW, placed, mode)
    out = run_mode(mode, monkeypatch, docs, sa, head, 16)
    assert out["big1"] == 0 and out["stats"]["fallback_elems"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("big", ["0", "31", "32", "63", "64", "100"])
def test_whole_warp_threshold(big, monkeypatch):
    """DSMFM_REFINE_BIG: below 32 the whole-warp ranking is off, 32..63 clamp to 64, above that it is the threshold;
    groups of 63, 64, 65 and 100 members on either side of each."""
    import dsmfm
    monkeypatch.setenv("DSMFM_REFINE_BIG", big)
    t = Text(5, 7)
    core = t.core(16)
    fams = [t.family(k, core) for k in (63, 64, 65, 100)]
    t.filler(KW)
    docs = t.docs()
    sa, head = layout(docs.size, KW, [(0, fams[0]), (100, fams[1]), (200, fams[2]), (300, fams[3])])
    out = run(docs, sa, head, 16, keep_sa=True)
    assert bool(out["paths"] & dsmfm.RPATH_COOP) == (int(big) >= 32)


# ---- window and warp ownership ----------------------------------------------------------------------------------

def _window_case(name, t):
    """(m, placed) of a named slot layout; members from t (depth 16 unless the case says otherwise)."""
    core = t.core(40)
    f = lambda k: t.family(k, core)
    if name == "heads_at_0_and_1023":
        return 3 * KW, [(0, f(40)), (KW - 1, f(40)), (2 * KW - 1, f(2))]
    if name == "last_group_768":
        return 3 * KW, [(KW - 1, f(GROUP_MAX))]
    if name == "last_group_769":
        return 3 * KW, [(KW - 1, f(GROUP_MAX + 1))]
    if name == "window_without_head":  # windows 1 .. 4 lie inside one group of 5000
        return 6 * KW, [(500, t.family(5000, t.core(60)))]
    if name == "warp_part_without_head":  # slots 128..255 (one warp's part) inside a group
        return KW, [(100, f(200)), (300, f(3))]
    if name == "straddle_127_128_129":
        return KW, [(100, f(27)), (127, f(2)), (129, f(3)), (255, f(2)), (383, f(130))]
    raise ValueError(name)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["heads_at_0_and_1023", "last_group_768", "last_group_769", "window_without_head",
                                  "warp_part_without_head", "straddle_127_128_129"])
def test_window_edges(name, mode, monkeypatch):
    t = Text(5, zlib.crc32(name.encode()) % 1000)
    m, placed = _window_case(name, t)
    docs, sa, head = state(t, m, placed, mode)
    out = run_mode(mode, monkeypatch, docs, sa, head, 16)
    st = out["stats"]
    if name == "last_group_768":
        assert st["fallback_elems"] == 0, "a last group of 768 members belongs to its window"
    if name == "last_group_769":
        assert out["big1"] == GROUP_MAX + 1, "a last group of 769 members takes the large-group path"
    if name == "window_without_head":
        assert st["fallback_elems"] >= 2 * 5000 and st["refine_launches"] >= 3, "the worklist carries the group"


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 2, 31, 33, 1000, 1024, 1025])
def test_range_sizes(m):
    """m at and around a head word and a window, and m not a multiple of 32; the last group ends at slot m - 1."""
    t = Text(5, m)
    core = t.core(16)
    placed = [] if m == 1 else [(max(0, m - min(m, 40)), t.family(min(m, 40), core))]
    if m > 100:
        placed.append((0, t.family(30, core)))
    t.filler(m)
    docs = t.docs()
    sa, head = layout(docs.size, m, placed)
    for keep in (True, False):
        run(docs, sa, head, 16, keep_sa=keep)


# ---- the large-group path -------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["one", "several", "several_rounds", "next_to_small"])
def test_large_groups(name, mode, monkeypatch):
    """One large group in a round; several (the second radix sort, by group id, runs); groups that stay larger than
    768 for several rounds (a long shared core, so the window worklist carries them); a large group between small
    ones in the same window."""
    import dsmfm
    t = Text(5, len(name))
    core = t.core(18)
    if name == "one":
        m, placed = 4 * KW, [(5, t.family(2000, core))]
    elif name == "several":  # the first group of 900 is not the last of its window: its CTA refines it
        m, placed = 5 * KW, [(0, t.family(900, core)), (1000, t.family(1200, t.core(18))), (2300, t.family(800, core))]
    elif name == "several_rounds":
        m, placed = 6 * KW, [(10, t.family(3000, t.core(120))), (3100, t.family(1500, t.core(80)))]
    else:
        m, placed = 2 * KW, [(100, t.family(5, core)), (110, t.family(10, core)), (200, t.family(1500, t.core(18)))]
    docs, sa, head = state(t, m, placed, mode)
    out = run_mode(mode, monkeypatch, docs, sa, head, 18)
    st = out["stats"]
    assert out["big1"] > 0
    assert bool(out["paths"] & dsmfm.RPATH_BIG_MULTI) == (name in ("several", "several_rounds"))
    if name == "several_rounds":
        assert st["refine_launches"] >= 4 and st["fallback_elems"] >= 3 * 4500


# ---- terminators ----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["keep_sa", "bwt_compact"])
@pytest.mark.parametrize("sigma", [5, 15, 255])
def test_terminator_at_every_offset(sigma, mode, monkeypatch):
    """Tails of 0 .. SPW + 1 symbols behind a core of 16 (the terminator at every offset of the next key and one
    past it), several documents per tail, some identical up to their terminator (they tie and keep text order
    although the documents behind them differ)."""
    spw = 64 // (3 if sigma <= 7 else (4 if sigma <= 15 else 8))
    t = Text(sigma, sigma)
    core = t.core(16)
    tails = [t.random(L, L, t.alpha[:2]) for L in range(spw + 2) for _ in range(3)]
    same = t.random(spw - 1, spw - 1, t.alpha[:2])
    fam_a = t.family(len(tails), core, tails=lambda i: tails[i])
    fam_b = t.family(40, core, tails=lambda i: same)  # 40 equal documents: tie through the terminator
    fam_c = t.family(200, core, tails=lambda i: tails[i % len(tails)])  # > 64 members: whole-warp ranking too
    docs, sa, head = state(t, 2 * KW, [(3, fam_a), (200, fam_b), (600, fam_c)], mode)
    run_mode(mode, monkeypatch, docs, sa, head, 16)


@pytest.mark.gpu
@pytest.mark.parametrize("keep", [True, False])
def test_one_symbol_documents(keep):
    """Documents of one symbol at depth 0: a group of every suffix of them, their terminators included (suffixes
    equal up to their terminator: they keep text order)."""
    t = Text(5, 3)
    for i in range(900):
        t.doc([t.alpha[i % 3]])
    docs = t.docs()
    first = 6  # behind the alphabet document
    mem = np.arange(first, docs.size)
    sa, head = layout(docs.size, docs.size, [(0, np.arange(first)), (first, mem)])
    run(docs, sa, head, 0, keep_sa=keep)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["candidate_terminated", "every_member_candidate", "no_member_candidate"])
@pytest.mark.parametrize("keep", [True, False])
def test_whole_warp_candidate(name, keep, monkeypatch):
    """The whole-warp ranking (DSMFM_REFINE_BIG=64) around a group's dominant key: a dominant key that is terminated
    (most members end right behind the core), one that every member carries (they differ only a window later), and
    groups of distinct keys where no key dominates."""
    import dsmfm
    monkeypatch.setenv("DSMFM_REFINE_BIG", "64")
    t = Text(5, len(name))
    core = t.core(16)
    two = t.alpha[:2]
    if name == "candidate_terminated":
        tails = lambda i: np.zeros(0, np.uint8) if i % 5 else t.random(1, 30, two)
    elif name == "every_member_candidate":
        common = t.random(30, 30)
        tails = lambda i: np.concatenate([common, t.random(0, 25, two)]).astype(np.uint8)
    else:
        tails = lambda i: t.random(25, 25)
    fams = [t.family(k, core, tails=tails) for k in (64, 100, 300)]
    t.filler(KW)
    docs = t.docs()
    sa, head = layout(docs.size, KW, [(0, fams[0]), (70, fams[1]), (200, fams[2])])
    out = run(docs, sa, head, 16, keep_sa=keep)
    assert out["paths"] & dsmfm.RPATH_COOP


# ---- compaction -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_compaction_word_and_tile_edges():
    """Mixed groups whose difference bits sit at bits 0 and 31 of a head word, and groups across the 8192-slot tiles
    of the compaction, among groups with a single BWT symbol."""
    import dsmfm
    t = Text(5, 11)
    core = t.core(16)
    mix = lambda k: t.family(k, core)
    uni = lambda k: t.family(k, core, x=t.alpha[1])
    a0, a1 = t.alpha[0], t.alpha[1]
    placed = [(30, t.family(2, core, x=[a0, a1])), (62, t.family(3, core, x=[a0, a1, a0])),
              (95, t.family(2, core, x=[a1, a0])), (200, uni(60)), (400, uni(300))]
    for edge in (TILE, 2 * TILE, 3 * TILE):
        placed += [(edge - 3, mix(7)), (edge + 40, uni(50)), (edge - 200, uni(100))]
    m = 3 * TILE + 500
    t.filler(m)
    docs = t.docs()
    sa, head = layout(docs.size, m, placed)
    out = run(docs, sa, head, 16)
    assert out["paths"] & dsmfm.RPATH_COMPACT


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["m_act_zero", "half", "half_plus_one"])
def test_compact_or_in_place(case):
    """No mixed group (nothing launched); mixed members exactly half of those in groups (dense copies); one more
    (refined in place)."""
    import dsmfm
    t = Text(5, 12)
    core = t.core(16)
    a, u = {"m_act_zero": (0, 80), "half": (40, 40), "half_plus_one": (41, 40)}[case]
    placed = [(100, t.family(u, core, x=t.alpha[2]))]
    if a:
        placed.append((300, t.family(a, core)))
    t.filler(KW)
    docs = t.docs()
    sa, head = layout(docs.size, KW, placed)
    out = run(docs, sa, head, 16)
    assert out["mixed"] == a
    assert bool(out["paths"] & dsmfm.RPATH_COMPACT) == (case == "half")
    if case == "m_act_zero":
        assert out["stats"]["refine_launches"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["scratch_alloc", "scratch_carved_dense_alloc", "dense_carved"])
def test_compaction_buffers(case):
    """The compaction scratch and the dense arrays carved out of the key buffers of the range, or allocated when the
    range is too small to hold them."""
    import dsmfm
    t = Text(5, 13)
    core = t.core(16)
    m, a, u = {"scratch_alloc": (32, 6, 20), "scratch_carved_dense_alloc": (256, 100, 120),
               "dense_carved": (4096, 100, 200)}[case]
    placed = [(0, t.family(a, core)), (a + 3, t.family(u, core, x=t.alpha[1]))]
    t.filler(m)
    docs = t.docs()
    sa, head = layout(docs.size, m, placed)
    out = run(docs, sa, head, 16)
    p = out["paths"]
    assert p & dsmfm.RPATH_COMPACT
    assert bool(p & dsmfm.RPATH_SCRATCH_ALLOC) == (case == "scratch_alloc")
    assert bool(p & dsmfm.RPATH_DENSE_ALLOC) == (case != "dense_carved")


# ---- every instantiation of the kernel ----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("lo_bits", [0, 10])
@pytest.mark.parametrize("coop", [False, True])
@pytest.mark.parametrize("keep", [True, False])
@pytest.mark.parametrize("sigma", [5, 15, 255])
def test_every_instantiation(sigma, keep, coop, lo_bits, monkeypatch):
    """BITS 3 / 4 / 8 x full or BWT order x whole-warp ranking on or off x u32 or split positions (lo_bits = 10:
    positions above 2^10 carry a high byte): the 24 instantiations of the refinement kernel, each asserted."""
    import dsmfm
    monkeypatch.setenv("DSMFM_REFINE_BIG", "64" if coop else "0")
    t = Text(sigma, sigma + 2)
    t.filler(3000)  # members above 2^10
    core = t.core(18)
    fams = [t.family(k, core) for k in (2, 40, 150, 900)]
    t.filler(2 * KW)
    docs = t.docs()
    assert np.unique(docs).size == sigma + 1
    sa, head = layout(docs.size, 3 * KW, [(5, fams[0]), (50, fams[1]), (200, fams[2]), (1900, fams[3])])
    out = run(docs, sa, head, 18, keep_sa=keep, lo_bits=lo_bits)
    p = out["paths"]
    assert bool(p & dsmfm.RPATH_COOP) == coop
    assert bool(p & dsmfm.RPATH_ORDER) == keep
    assert bool(p & dsmfm.RPATH_WIDE) == (lo_bits > 0)
    assert (p >> dsmfm.RPATH_BITS_SHIFT) & 15 == {5: 3, 15: 4, 255: 8}[sigma]
    assert out["big1"] > 0


# ---- the build's own state ----------------------------------------------------------------------------------------

def _build_docs(kind):
    if kind == "reads":
        import dsmgen
        return dsmgen.docs(seed=5, pool_seed=5, pool_size=2, n_genomes=2, genome_len=20000, n_reads=4000,
                           read_len=100, sub=0.005, pn=0.001)
    t = Text({"4bit": 12, "8bit": 200}.get(kind, 5), 21)
    if kind == "poly_a":
        t.doc(np.full(5000, t.alpha[0]))
        for _ in range(200):
            t.doc(np.full(40, t.alpha[0]))
    elif kind == "duplicates":
        d = [t.random(5, 90) for _ in range(3)]
        for i in range(300):
            t.doc(d[i % 3])
    else:
        t.filler(100_000, 1, 200)
    return t.docs()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["reads", "poly_a", "duplicates", "4bit", "8bit"])
def test_state_of_the_initial_sort(kind):
    """initial_sort -> refine from its heads at its first-key depth gives the suffix array of a build with
    FLAG_KEEP_SA and the oracle's, and in BWT order the oracle's BWT: the entry point runs what the build runs."""
    import dsmfm
    import oracle
    docs = _build_docs(kind)
    init = dsmfm.initial_sort(docs)
    assert init["carry"] == 1
    want_bwt, want_sa = oracle.bwt(docs.tobytes(), want_sa=True)
    with dsmfm.Builder(flags=dsmfm.FLAG_KEEP_SA) as b:
        b.append_batch(docs)
        b.finish()
        built = b.suffix_array()
    full = dsmfm.refine(docs, init["sa"], init["head"], init["first_syms"], keep_sa=True)
    assert np.array_equal(full["sa"], built.astype(np.uint64))
    assert np.array_equal(full["sa"], want_sa)
    assert full["bwt"].tobytes() == want_bwt
    assert full["stats"]["active"][0] == init["remaining"]
    part = dsmfm.refine(docs, init["sa"], init["head"], init["first_syms"])
    assert part["bwt"].tobytes() == want_bwt


# ---- beyond one scan block of the compaction ------------------------------------------------------------------

@pytest.mark.gpu
def test_more_than_one_scan_block():
    """m > 2^26 slots (more than 8192 compaction tiles: the scan of the tile counts carries across its blocks) with
    3000 scattered mixed groups and as many with a single BWT symbol (so the mixed ones are compacted), checked
    group by group.  Host memory: about 5 GB."""
    import dsmfm
    if os.environ.get("DSMFM_TEST_SMALL"):
        pytest.skip("needs more than 2^26 slots")
    m = (1 << 26) + 300_000
    rng = np.random.default_rng(26)
    t = Text(5, 26)
    core = t.core(16)
    sizes = rng.integers(2, 40, size=3000)
    fams = [t.family(int(k), core) for k in sizes] + [t.family(int(k), core, x=t.alpha[0]) for k in sizes]
    # fillers: one random text of m symbols cut into documents of 1..150 symbols
    body = rng.choice(t.alpha, size=m).astype(np.uint8)
    ends = np.cumsum(rng.integers(2, 152, size=m // 50)) - 1
    body[ends[ends < m - 2]] = 0
    body[-1] = 0
    docs = np.concatenate([t.docs(), body])
    del body
    slots = np.sort(rng.choice(np.arange(0, m - 64, 64), size=len(fams), replace=False))
    sa, head = layout(docs.size, m, list(zip(slots, fams)))
    out = run(docs, sa, head, 16, rank=None)
    assert out["paths"] & dsmfm.RPATH_COMPACT
    assert out["mixed"] > 0


# ---- the entry point refuses states the build could not reach (no GPU needed) ----------------------------------

def _refusal(case):
    docs = np.frombuffer(b"ACGTACGT\0GATTACA\0ACGTACGA\0" * 4, np.uint8).copy()
    n = docs.size
    sa = np.arange(n, dtype=np.uint64)
    head = pack_bits(np.ones(n, bool))
    kw = dict(depth=0, keep_sa=False, lo_bits=0)
    if case == "empty_doc":
        docs = np.concatenate([docs[:9], [0], docs[9:]]).astype(np.uint8)  # behind the terminator at 8
    elif case == "unterminated":
        docs = docs[:-1].copy()
        sa, head = sa[:-1], pack_bits(np.ones(n - 1, bool))
    elif case == "m_zero":
        sa = sa[:0]
    elif case == "m_above_n":
        # (more than n distinct positions below n do not exist: the extra entry necessarily breaks a position rule
        # too; the entry point refuses m > n before it reads any position)
        sa = np.append(sa, 0).astype(np.uint64)
        head = pack_bits(np.ones(n + 1, bool))
    elif case == "position_past_text":
        sa[3] = n
    elif case == "position_twice":
        sa[3] = 4
    elif case == "head_bit_0_clear":
        f = np.ones(n, bool)
        f[0] = False
        head = pack_bits(f)
    elif case == "group_not_ascending":  # slots 0, 1: positions 18, 1 at depth 0
        sa[0], sa[18] = 18, 0
        f = np.ones(n, bool)
        f[1] = False
        head = pack_bits(f)
    elif case in ("members_differ", "terminator_within_depth", "depth_ok"):
        # slots 0, 1 form a group: positions 0 and 17 share "ACGTACG" (7 symbols) and differ at the 8th; positions
        # 8 and 16 are terminators (they tie at depth 1 only by reaching their terminator)
        p, q = (8, 16) if case == "terminator_within_depth" else (0, 17)
        sa[[0, p]], sa[[1, q]] = sa[[p, 0]], sa[[q, 1]]
        f = np.ones(n, bool)
        f[1] = False
        head = pack_bits(f)
        kw["depth"] = {"members_differ": 8, "depth_ok": 7, "terminator_within_depth": 1}[case]
    elif case == "lo_bits_3":
        kw["lo_bits"] = 3
    elif case == "lo_bits_33":
        kw["lo_bits"] = 33
    elif case == "position_beyond_lo_bits":
        kw["lo_bits"] = 4  # positions below 2^12 only
        big = np.concatenate([docs] * 200)
        docs = big
        sa = np.arange(big.size, dtype=np.uint64)
        head = pack_bits(np.ones(big.size, bool))
    return docs, sa, head, kw


REFUSALS = ["empty_doc", "unterminated", "m_zero", "m_above_n", "position_past_text", "position_twice",
            "head_bit_0_clear", "group_not_ascending", "members_differ", "terminator_within_depth", "lo_bits_3",
            "lo_bits_33", "position_beyond_lo_bits", "unknown_flags"]


@pytest.mark.parametrize("case", REFUSALS)
def test_refine_refuses_unreachable_state(case):
    import ctypes as C
    import dsmfm
    L = dsmfm.lib()
    docs, sa, head, kw = _refusal(case)
    flags = 4 if case == "unknown_flags" else 0
    m = sa.size
    sa_out, bwt_out = np.zeros(max(1, m), np.uint64), np.zeros(max(1, m), np.uint8)
    st, paths = dsmfm.Stats(), C.c_uint32()
    rc = L.dsmfm_dbg_refine(0, docs.ctypes.data, docs.size, sa.ctypes.data if m else sa_out.ctypes.data,
                            head.ctypes.data, m, kw["depth"], flags, kw["lo_bits"], sa_out.ctypes.data,
                            bwt_out.ctypes.data, C.byref(st), C.byref(paths))
    assert rc == dsmfm.EINVAL


@pytest.mark.parametrize("case", ["depth_ok", "position_beyond_lo_bits_ok"])
def test_refine_refusal_cases_are_minimal(case):
    """The states next to the refused ones pass the checks: they fail only where a device is needed, or run."""
    import dsmfm
    if case == "depth_ok":
        docs, sa, head, kw = _refusal("depth_ok")
    else:
        docs, sa, head, kw = _refusal("position_beyond_lo_bits")
        sa, kw["lo_bits"] = sa[:1 << 12], 4
        head = pack_bits(np.ones(sa.size, bool))
    try:
        dsmfm.refine(docs, sa, head, kw["depth"], lo_bits=kw["lo_bits"])
    except dsmfm.DsmfmError as e:
        assert e.code != dsmfm.EINVAL
