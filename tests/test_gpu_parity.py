"""GPU suite: the CUDA path, called through the C ABI (libdsmfm.so), against the oracle and the
golden files of the unmodified reference.  Bit-exact everywhere (integer / byte work)."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import cases
import oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MANIFEST = json.load(open(os.path.join(GOLDEN, "manifest.json")))


def _golden(name, ext):
    with open(os.path.join(GOLDEN, name + ext), "rb") as f:
        return f.read()


def _build(docs, **kw):
    import dsmfm
    return dsmfm.build_fmi(docs, **kw)


def _assert_same_fmi(got, want):
    assert oracle.diff_fmi(got, want) == []
    assert got == want


# ---- kernels in isolation -------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 31, 4095, 4096, 4097, 100_003, 3_000_000])
@pytest.mark.parametrize("bits", [(0, 64), (0, 63), (3, 19), (0, 5)])
def test_radix_sort_matches_stable_numpy_sort(n, bits):
    import dsmfm
    rng = np.random.default_rng(n * 131 + bits[1])
    keys = rng.integers(0, 2**64, size=n, dtype=np.uint64)
    if n > 1000:  # plant long runs of equal keys to exercise stability
        keys[: n // 3] = keys[0]
    vals = np.arange(n, dtype=np.uint32)
    lo, hi = bits
    mask = np.uint64(((1 << (hi - lo)) - 1) << lo) if hi - lo < 64 else np.uint64(2**64 - 1)
    order = np.argsort(keys & mask, kind="stable")
    k, v = keys.copy(), vals.copy()
    dsmfm.radix_sort(k, v, lo, hi)
    assert np.array_equal(v, vals[order])
    assert np.array_equal(k, keys[order])


@pytest.mark.parametrize("bits", [(0, 48), (0, 24), (0, 60), (3, 39), (12, 48)])
@pytest.mark.parametrize("n,dna", [(1, True), (4097, True), (1_000_003, True), (600_000, False)])
def test_radix_sort_key_widths_of_the_build(n, dna, bits):
    """The key widths the build uses (48 bits = 16 three-bit symbols, and the other multiples of a symbol), on
    DNA-like keys (few digit values, long runs) and on random keys."""
    import dsmfm
    rng = np.random.default_rng(n + bits[1])
    if dna:
        sym = rng.choice(np.array([0, 1, 2, 3, 4, 5, 6], dtype=np.uint64), size=(n, 21), p=[.02, .02, .235, .235, .235, .02, .235])
        keys = np.zeros(n, dtype=np.uint64)
        for j in range(21):
            keys = (keys << np.uint64(3)) | sym[:, j]
    else:
        keys = rng.integers(0, 2**64, size=n, dtype=np.uint64)
    if n > 1000:
        keys[: n // 4] = keys[0]
    vals = np.arange(n, dtype=np.uint32)
    lo, hi = bits
    mask = np.uint64(((1 << (hi - lo)) - 1) << lo)
    order = np.argsort(keys & mask, kind="stable")
    k, v = keys.copy(), vals.copy()
    dsmfm.radix_sort(k, v, lo, hi)
    assert np.array_equal(v, vals[order])
    assert np.array_equal(k, keys[order])


def test_radix_sort_dna_like_keys():
    """3-bit symbols, only 5 of 8 codes in use: the skewed digit histograms of the real workload."""
    import dsmfm
    rng = np.random.default_rng(7)
    n = 1_500_000
    sym = rng.choice(np.array([2, 3, 4, 6], dtype=np.uint64), size=(n, 21))
    keys = np.zeros(n, dtype=np.uint64)
    for j in range(21):
        keys = (keys << np.uint64(3)) | sym[:, j]
    vals = np.arange(n, dtype=np.uint32)
    order = np.argsort(keys, kind="stable")
    k, v = keys.copy(), vals.copy()
    dsmfm.radix_sort(k, v, 0, 63)
    assert np.array_equal(v, vals[order])


@pytest.mark.parametrize("alpha,n", [(b"\0-ACGNT", 1), (b"\0-ACGNT", 63), (b"\0-ACGNT", 64), (b"\0-ACGNT", 8191),
                                     (b"\0-ACGNT", 8192), (b"\0-ACGNT", 300_001), (b"A", 1000), (b"AB", 5000),
                                     (bytes(range(256)), 70_000), (b"\0-.0123ACGNT", 50_000)])
def test_wavelet_tree_and_bitrank_match_oracle(alpha, n):
    import dsmfm
    rng = np.random.default_rng(n)
    # skewed symbol frequencies, like a BWT of reads
    w = rng.random(len(alpha)) ** 3 + 1e-3
    seq = np.frombuffer(alpha, dtype=np.uint8)[rng.choice(len(alpha), size=n, p=w / w.sum())]
    got = dsmfm.wavelet_fmi(seq)
    want = oracle.fmi_from_bwt(seq.tobytes(), 124, 0, 0)
    _assert_same_fmi(got, want)


# ---- the whole path against the reference's golden files -------------------------------------------

@pytest.mark.parametrize("name", sorted(MANIFEST["files"]))
def test_build_matches_reference_golden_file(name):
    docs, nd = oracle.fasta_to_docs(_golden(name, ".fasta"))
    _assert_same_fmi(_build(docs), _golden(name, ".fmi"))


def test_samplerate_option():
    docs, _ = oracle.fasta_to_docs(_golden("small_random", ".fasta"))
    assert _build(docs, samplerate=32) == _golden("small_random", ".s32.fmi")


@pytest.mark.parametrize("name", sorted(MANIFEST["digests"]))
def test_build_matches_reference_digest(name):
    docs, _ = oracle.fasta_to_docs(cases.digest_cases()[name])
    got = _build(docs)
    assert len(got) == MANIFEST["digests"][name]["fmi_bytes"]
    assert hashlib.sha256(got).hexdigest() == MANIFEST["digests"][name]["fmi_sha256"]


@pytest.mark.parametrize("name", sorted(MANIFEST["generated"]))
def test_build_matches_reference_on_generated_reads(name):
    import dsmgen
    g = MANIFEST["generated"][name]
    got = _build(dsmgen.docs(**g["params"]))
    assert len(got) == g["fmi_bytes"]
    assert hashlib.sha256(got).hexdigest() == g["fmi_sha256"]


# ---- against the oracle on seeded inputs, including the intermediate products ------------------------

@pytest.mark.parametrize("seed,kw", [
    (1, dict(nreads=500, maxlen=100, genome=2000)),
    (2, dict(nreads=3000, maxlen=60, minlen=60, genome=500, dup=0.0, pn=0.0)),   # deep ties
    (3, dict(nreads=800, maxlen=300, genome=1200, dup=0.4)),                     # long ragged reads
    (4, dict(nreads=2500, maxlen=45, alpha="A", genome=64)),                     # groups beyond one CTA
    (5, dict(nreads=700, maxlen=80, alpha="ACGT0123.", genome=900)),             # 4 bits per symbol
])
def test_suffix_array_bwt_and_index_match_oracle(seed, kw):
    """Seed 4 has groups too large for a CTA: they go through the large-group path and come back to their windows
    in a later refinement launch (the window worklist)."""
    import dsmfm
    docs, nd = oracle.fasta_to_docs(cases.rnd_fasta(seed, **kw))
    want_bwt, want_sa = oracle.bwt(docs, want_sa=True)
    with dsmfm.Builder(flags=dsmfm.FLAG_KEEP_BWT | dsmfm.FLAG_KEEP_SA) as b:
        b.append_batch(docs)
        idx = b.finish()
        assert idx.n == len(docs) and idx.number_of_texts == nd
        assert idx.max_text_length == oracle.doc_stats(docs)[1]
        sa = b.suffix_array()
        bad = np.nonzero(sa.astype(np.uint64) != want_sa)[0]
        assert bad.size == 0, "first suffix-array mismatch at rank %d" % bad[0]
        assert b.bwt() == want_bwt
        _assert_same_fmi(b.fmi(), oracle.fmi_from_docs(docs))
        if seed == 4:
            assert b.stats().refine_launches >= 2


def test_long_first_key_of_large_collections(monkeypatch):
    """Collections beyond 3.5 G symbols sort 18 symbols (54 bits, 7 passes) instead of 16; with the threshold moved
    down the same schedule runs on small inputs, unsharded and as key-range shards with wide positions."""
    import dsmfm
    monkeypatch.setenv("DSMFM_LONG_KEY_ABOVE", "1000")
    for name in ["reads100", "poly_a", "duplicates", "mixed_alphabet"]:
        docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
        _assert_same_fmi(_build(docs), _golden(name, ".fmi"))
    docs, _ = oracle.fasta_to_docs(cases.digest_cases()["reads100_3k"])
    with dsmfm.Builder(device=0) as b:
        b.append_batch(docs)
        b.finish()
        assert b.stats().sort_passes == 7
        assert hashlib.sha256(b.fmi()).hexdigest() == MANIFEST["digests"]["reads100_3k"]["fmi_sha256"]
    monkeypatch.setenv("DSMFM_POS_LO_BITS", "12")
    want_bwt, want_sa = oracle.bwt(docs, want_sa=True)
    fmi, bwt, sa = _sharded_build(docs, 3)
    assert bwt == want_bwt and np.array_equal(sa.astype(np.uint64), want_sa)
    assert hashlib.sha256(fmi).hexdigest() == MANIFEST["digests"]["reads100_3k"]["fmi_sha256"]


@pytest.mark.parametrize("first_key_bits", ["63", "24", "9"])
def test_first_key_width_does_not_change_the_result(first_key_bits, monkeypatch):
    """The initial sort may use fewer symbols (more refinement) or all 21 (BWT gathered instead of
    carried through the sort): the index is the same."""
    monkeypatch.setenv("DSMFM_FIRST_KEY_BITS", first_key_bits)
    for name in ["reads100", "poly_a", "duplicates"]:
        docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
        _assert_same_fmi(_build(docs), _golden(name, ".fmi"))


@pytest.mark.parametrize("env", [{"DSMFM_REFINE_COMPACT": "0"}, {"DSMFM_REFINE_FULL_ORDER": "1"},
                                 {"DSMFM_REFINE_BIG": "64"}, {"DSMFM_REFINE_BIG": "64", "DSMFM_REFINE_COMPACT": "0"},
                                 {"DSMFM_REFINE_BIG": "0", "DSMFM_REFINE_COMPACT": "0"},
                                 {"DSMFM_REFINE_BIG": "64", "DSMFM_REFINE_FULL_ORDER": "1"}])
def test_refinement_schedules_give_the_same_index(monkeypatch, env):
    """BWT-only refinement on dense copies of the mixed groups (default), in place with the difference bitmap, and
    the full suffix order, each with both ranking schemes of the refinement kernel (whole groups per warp-load with
    match.any, and large groups by the whole warp around their dominant key): one index."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for name in ("reads100", "duplicates", "poly_a", "mixed_alphabet", "one_base_reads"):
        docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
        _assert_same_fmi(_build(docs), _golden(name, ".fmi"))
    for name in ("high_coverage", "ragged_2k"):
        docs, _ = oracle.fasta_to_docs(cases.digest_cases()[name])
        got = _build(docs)
        assert hashlib.sha256(got).hexdigest() == MANIFEST["digests"][name]["fmi_sha256"]


def test_bwt_only_build_sorts_fewer_suffixes():
    """The statistics tell the two refinements apart: members sorted vs members of tie groups."""
    import dsmfm
    import dsmgen
    docs = dsmgen.docs(**MANIFEST["generated"]["gen_20k"]["params"])
    with dsmfm.Builder(device=0) as b:
        b.append_batch(docs)
        b.finish()
        lean = b.stats()
        fmi = b.fmi()
    with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA) as b:
        b.append_batch(docs)
        b.finish()
        full = b.stats()
        assert b.fmi() == fmi
    assert full.refine_members == full.active[0] > 0
    assert 0 < lean.refine_members < full.refine_members // 2
    assert lean.refine_key_fetches < full.refine_key_fetches


def test_arbitrary_byte_alphabet():
    """TextCollectionBuilder admits any byte 1..255 (TextCollectionBuilder.h:52): 8 bits per symbol."""
    rng = np.random.default_rng(11)
    parts = []
    for _ in range(300):
        ln = int(rng.integers(1, 120))
        parts.append(rng.integers(1, 256, size=ln, dtype=np.uint8).tobytes() + b"\0")
    docs = b"".join(parts)
    _assert_same_fmi(_build(docs), oracle.fmi_from_docs(docs))


def test_insert_text_one_by_one_equals_batch():
    import dsmfm
    docs, nd = oracle.fasta_to_docs(_golden("reads100", ".fasta"))
    with dsmfm.Builder() as b:
        for d in docs.split(b"\0")[:-1]:
            b.insert_text(d)
        b.finish()
        assert b.fmi() == _golden("reads100", ".fmi")


def test_error_behaviour():
    import dsmfm
    with dsmfm.Builder() as b:
        with pytest.raises(dsmfm.DsmfmError) as e:
            b.insert_text(b"")                       # TextCollectionBuilder.cpp:86-91
        assert e.value.code == dsmfm.EEMPTY
    with dsmfm.Builder() as b:
        b.append_batch(b"AC\0\0GT\0")                # empty document inside a batch
        with pytest.raises(dsmfm.DsmfmError) as e:
            b.finish()
        assert e.value.code == dsmfm.EEMPTY
    with dsmfm.Builder() as b:
        with pytest.raises(dsmfm.DsmfmError) as e:
            b.append_batch(b"ACGT")                  # unterminated
        assert e.value.code == dsmfm.EINVAL
    with dsmfm.Builder() as b:
        b.append_batch(b"ACGT\0")
        b.finish()
        with pytest.raises(dsmfm.DsmfmError) as e:   # TextCollectionBuilder.cpp:67-71
            b.insert_text(b"AC")
        assert e.value.code == dsmfm.EINVAL


def test_stats_are_reported():
    import dsmfm
    import dsmgen
    kw = MANIFEST["generated"]["gen_20k"]["params"]
    with dsmfm.Builder() as b:
        b.append_batch(dsmgen.docs(**kw))
        b.finish()
        s = b.stats()
        assert s.n == 20_000 * 202 and s.bases == 20_000 * 201
        assert s.bits_per_symbol == 3 and s.sigma == 6
        assert s.sort_passes == 6 and s.kernel_launches > 10
        assert s.rounds >= 1 and s.active[0] > 0
        assert s.ms_total > 0 and s.ms_sort_pass > 0


# ---- the drop-in CLI ----------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["empty", "multiline_and_blank", "no_trailing_newline", "crlf", "reads100",
                                  "mixed_alphabet"])
def test_builder_cli_writes_the_reference_bytes(name, tmp_path):
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    fa = tmp_path / (name + ".fasta")
    fa.write_bytes(_golden(name, ".fasta"))
    r = subprocess.run([exe, "-v", str(fa)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(str(fa) + ".fmi", "rb").read()
    _assert_same_fmi(got, _golden(name, ".fmi"))
    # explicit output name and stdin input (builder.cpp:396-397, 426-427)
    r = subprocess.run([exe, "-", str(tmp_path / "out")], input=_golden(name, ".fasta"), capture_output=True)
    assert r.returncode == 0, r.stderr
    assert open(str(tmp_path / "out.fmi"), "rb").read() == _golden(name, ".fmi")
    # the reference's per-read loop on the host (one InsertText per read) instead of the GPU front end
    r = subprocess.run([exe, "--host-parse", str(fa), str(tmp_path / "hp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(str(tmp_path / "hp.fmi"), "rb").read() == _golden(name, ".fmi")
    if name in ("crlf", "multiline_and_blank"):
        assert "contains invalid symbol(s)" in r.stderr


def test_builder_cli_streams_the_input_in_pieces(tmp_path):
    """A 1 MB input buffer (DSMFM_FASTA_CHUNK_MB) makes the CLI hand the file to the GPU front end in pieces cut at
    header lines; the index must not depend on it."""
    import dsmfm
    import dsmgen
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    kw = dict(seed=5, pool_seed=5, pool_size=2, n_genomes=2, genome_len=20000, n_reads=40000, read_len=100, sub=0.005, pn=0.001)
    fa = tmp_path / "s.fasta"
    dsmgen.fasta(**kw).tofile(str(fa))
    env = dict(os.environ, DSMFM_FASTA_CHUNK_MB="1")
    r = subprocess.run([exe, "-v", str(fa)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    assert r.stderr.count("Inserting:") >= 4
    assert open(str(fa) + ".fmi", "rb").read() == dsmfm.build_fmi(dsmgen.docs(**kw))


@pytest.mark.parametrize("gpus", [2, 3, 8])
@pytest.mark.parametrize("name", ["empty", "multiline_and_blank", "no_trailing_newline", "reads100", "mixed_alphabet", "single"])
def test_builder_cli_on_several_gpus_writes_the_reference_bytes(name, gpus, tmp_path):
    """`builder --gpus N` (host/MultiGpuBuilder.cpp: one host thread per rank, packed slots exchanged by peer
    copies, every rank writes its share of the file).  Rank r runs on device r modulo the devices present, so the
    N-rank build is checked on a one-GPU box as well; the file must be the reference's, byte for byte."""
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    fa = tmp_path / (name + ".fasta")
    fa.write_bytes(_golden(name, ".fasta"))
    r = subprocess.run([exe, "-v", "--gpus", str(gpus), str(fa)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    _assert_same_fmi(open(str(fa) + ".fmi", "rb").read(), _golden(name, ".fmi"))
    r = subprocess.run([exe, "--gpus", str(gpus), "-s", "32", "-", str(tmp_path / "out")], input=_golden(name, ".fasta"),
                       capture_output=True)
    assert r.returncode == 0, r.stderr
    if name == "small_random":
        assert open(str(tmp_path / "out.fmi"), "rb").read() == _golden("small_random", ".s32.fmi")


def test_builder_cli_on_several_gpus_matches_one_gpu_on_a_generated_sample(tmp_path):
    import dsmgen
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    kw = MANIFEST["generated"]["gen_20k"]["params"]
    fa = tmp_path / "g.fasta"
    dsmgen.fasta(**kw).tofile(str(fa))
    r = subprocess.run([exe, "-v", "--gpus", "4", str(fa), str(tmp_path / "four")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "rank 3" in r.stderr
    got = open(str(tmp_path / "four.fmi"), "rb").read()
    import hashlib
    assert hashlib.sha256(got).hexdigest() == MANIFEST["generated"]["gen_20k"]["fmi_sha256"]


def test_builder_cli_samplerate(tmp_path):
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    fa = tmp_path / "s.fasta"
    fa.write_bytes(_golden("small_random", ".fasta"))
    subprocess.run([exe, "-s", "32", str(fa)], check=True, capture_output=True)
    assert open(str(fa) + ".fmi", "rb").read() == _golden("small_random", ".s32.fmi")


# ---- live differential runs when the compiled reference travelled with the snapshot --------------------

@pytest.mark.skipif(not oracle.have_reference(), reason="oracle/_ref not present")
def test_toydata_shaped_sample_matches_live_reference(tmp_path):
    """A 60k-read toydata-shaped sample through both builders (the reference needs ~8 s for it)."""
    import dsmgen
    kw = dict(seed=31, pool_seed=99, pool_size=16, n_genomes=10, genome_len=60_000, n_reads=60_000, read_len=100,
              sub=0.005, pn=0.001)
    fasta = dsmgen.fasta(**kw).tobytes()
    want = oracle.reference_build(fasta, tmp_path)
    _assert_same_fmi(_build(dsmgen.docs(**kw)), want)


# ---- one collection cut into key ranges (the multi-GPU path, here with every range on one device) ------

def _sharded_build(docs, shard_count, span=1, pieces=False):
    """Builds every slice of the global suffix order with its own builder, concatenates the BWT slices
    on the device and assembles the index on the first builder.  Returns (fmi, bwt, sa)."""
    import torch
    import dsmfm
    builders, bw, sa, nxt = [], [], [], 0
    try:
        for first in range(0, shard_count, span):
            b = dsmfm.Builder(flags=dsmfm.FLAG_KEEP_SA, shard_index=first, shard_count=shard_count,
                              shard_span=min(span, shard_count - first))
            builders.append(b)
            b.append_batch(docs)
            b.build_device()
            info = b.shard_info()
            assert info.n_total == len(docs)
            assert info.rank_begin == nxt, "slices are not contiguous"
            nxt += info.count
            bw.append(torch.empty(info.count, dtype=torch.uint8, device="cuda"))
            sa.append(torch.empty(info.count, dtype=torch.int64, device="cuda"))
            b.shard_export(bw[-1], sa[-1])
        assert nxt == len(docs)
        full = torch.cat(bw)
        if pieces:  # every slice contributes its bits of every wavelet-tree node; the first builder merges them
            hist_all = np.stack([b.slice_hist() for b in builders])
            assert np.array_equal(hist_all.sum(axis=0), np.bincount(np.frombuffer(docs, dtype=np.uint8), minlength=256))
            bufs = []
            for r, b in enumerate(builders):
                bufs.append(torch.empty(b.pieces_bytes(hist_all, r), dtype=torch.uint8, device="cuda"))
                b.build_pieces(hist_all, r, bufs[-1])
            allp = torch.cat(bufs)
            assert allp.numel() == builders[0].pieces_bytes(hist_all, len(builders))
            builders[0].assemble_pieces(hist_all, allp)
        else:
            builders[0].assemble(full, len(docs))
        builders[0].fetch()
        return builders[0].fmi(), full.cpu().numpy().tobytes(), torch.cat(sa).cpu().numpy()
    finally:
        for b in builders:
            b.close()


@pytest.mark.parametrize("shards,span", [(2, 1), (3, 1), (8, 1), (8, 4), (5, 2), (64, 16)])
@pytest.mark.parametrize("name", ["reads100", "poly_a", "duplicates", "mixed_alphabet", "one_base_reads", "single"])
def test_key_range_shards_concatenate_to_the_reference_index(name, shards, span):
    docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
    want_bwt, want_sa = oracle.bwt(docs, want_sa=True)
    fmi, bwt, sa = _sharded_build(docs, shards, span)
    assert np.array_equal(sa.astype(np.uint64), want_sa)
    assert bwt == want_bwt
    _assert_same_fmi(fmi, _golden(name, ".fmi"))


@pytest.mark.parametrize("lo_bits", ["12", "15"])
def test_wide_positions_on_small_inputs(monkeypatch, lo_bits):
    """Collections beyond 2^32 symbols keep the high part of a text position in the key's spare bits and
    then in a byte array next to the suffix array; DSMFM_POS_LO_BITS shrinks the low part so that the
    same code runs on inputs the oracle can check."""
    monkeypatch.setenv("DSMFM_POS_LO_BITS", lo_bits)
    for name, shards, span in [("reads100", 3, 1), ("poly_a", 2, 1), ("colour_space", 4, 2), ("two_letter", 2, 2)]:
        docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
        want_bwt, want_sa = oracle.bwt(docs, want_sa=True)
        fmi, bwt, sa = _sharded_build(docs, shards, span)
        assert np.array_equal(sa.astype(np.uint64), want_sa)
        assert bwt == want_bwt
        _assert_same_fmi(fmi, _golden(name, ".fmi"))
    docs, _ = oracle.fasta_to_docs(cases.digest_cases()["high_coverage"])
    fmi, _, _ = _sharded_build(docs, 3, 1)
    assert hashlib.sha256(fmi).hexdigest() == MANIFEST["digests"]["high_coverage"]["fmi_sha256"]


def test_sharded_arbitrary_byte_alphabet(monkeypatch):
    monkeypatch.setenv("DSMFM_POS_LO_BITS", "10")
    rng = np.random.default_rng(12)
    docs = b"".join(rng.integers(1, 256, size=int(rng.integers(1, 90)), dtype=np.uint8).tobytes() + b"\0"
                    for _ in range(200))
    fmi, bwt, sa = _sharded_build(docs, 3, 1)
    want_bwt, want_sa = oracle.bwt(docs, want_sa=True)
    assert np.array_equal(sa.astype(np.uint64), want_sa) and bwt == want_bwt
    _assert_same_fmi(fmi, oracle.fmi_from_docs(docs))


def test_sharded_builder_errors():
    import dsmfm
    with pytest.raises(dsmfm.DsmfmError):
        dsmfm.Builder(shard_index=2, shard_count=2)
    with pytest.raises(dsmfm.DsmfmError):
        dsmfm.Builder(shard_index=1, shard_count=4, shard_span=4)
    with dsmfm.Builder(shard_index=0, shard_count=2) as b:
        b.append_batch(b"ACGT\0")
        b.build_device()
        with pytest.raises(dsmfm.DsmfmError):   # a slice is not an index
            b.fetch()


@pytest.mark.parametrize("shards,span", [(2, 1), (3, 1), (8, 2), (37, 1)])
@pytest.mark.parametrize("name", ["reads100", "poly_a", "duplicates", "mixed_alphabet", "one_base_reads", "single",
                                  "two_letter", "empty"])
def test_wavelet_tree_assembled_from_per_slice_pieces(name, shards, span):
    """The multi-GPU wavelet tree: every slice's bits are built at their global bit offset and merged."""
    docs, _ = oracle.fasta_to_docs(_golden(name, ".fasta"))
    if not docs:
        pytest.skip("the empty collection is built unsharded")
    fmi, _, _ = _sharded_build(docs, shards, span, pieces=True)
    _assert_same_fmi(fmi, _golden(name, ".fmi"))


def test_pieces_on_a_generated_sample():
    import dsmgen
    g = MANIFEST["generated"]["gen_20k"]
    fmi, _, _ = _sharded_build(dsmgen.docs(**g["params"]).tobytes(), 5, 1, pieces=True)
    assert hashlib.sha256(fmi).hexdigest() == g["fmi_sha256"]


# ---- suffix-array samples: the `.sa` file of the reference's dormant FMIndex::saveSamples -----------------

def _sa_file(docs, samplerate):
    import dsmfm
    with dsmfm.Builder(flags=dsmfm.FLAG_KEEP_SA, samplerate=samplerate) as b:
        if len(docs):
            b.append_batch(docs)
        b.finish()
        return b.sa_file(), b.fmi()


@pytest.mark.parametrize("fn", sorted(MANIFEST["sa"]))
def test_sa_file_matches_reference_golden(fn):
    e = MANIFEST["sa"][fn]
    docs, _ = oracle.fasta_to_docs(_golden(e["case"], ".fasta"))
    got, _ = _sa_file(docs, e["samplerate"])
    assert got == _golden(fn, "")


@pytest.mark.parametrize("key", sorted(MANIFEST["sa_digests"]))
def test_sa_file_matches_reference_digest(key):
    e = MANIFEST["sa_digests"][key]
    docs, _ = oracle.fasta_to_docs(cases.digest_cases()[e["case"]])
    got, _ = _sa_file(docs, e["samplerate"])
    assert len(got) == e["bytes"] and hashlib.sha256(got).hexdigest() == e["sha256"]


def test_sa_file_on_generated_reads_and_empty_collection():
    import dsmgen
    g = MANIFEST["generated"]["gen_20k"]
    got, fmi = _sa_file(dsmgen.docs(**g["params"]).tobytes(), 0)
    assert hashlib.sha256(fmi).hexdigest() == g["fmi_sha256"]
    assert len(got) == g["sa_bytes"] and hashlib.sha256(got).hexdigest() == g["sa_sha256"]
    got, _ = _sa_file(b"", 124)
    assert got == oracle.sa_file_from_docs(b"", 124)


def test_sa_file_needs_the_suffix_array():
    import dsmfm
    with dsmfm.Builder() as b:
        b.append_batch(b"ACGT\0")
        b.finish()
        with pytest.raises(dsmfm.DsmfmError) as e:
            b.sa_file()
        assert e.value.code == dsmfm.EINVAL


def test_builder_cli_samples_option(tmp_path):
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    fa = tmp_path / "r.fasta"
    fa.write_bytes(_golden("reads100", ".fasta"))
    r = subprocess.run([exe, "--samples", "-s", "16", str(fa)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(str(fa) + ".sa", "rb").read() == _golden("reads100.s16", ".sa")


# ---- BASELINE.json configs[1]: several samples, then the reference's own mining pipeline on both sets of indexes ----

@pytest.mark.skipif(not oracle.have_reference(), reason="oracle/_ref not present")
def test_five_samples_and_identical_mining_output(tmp_path):
    """Five toydata-shaped samples (SURVEY 8d C2: each draws 10 genomes of a shared pool of 16) are built by the
    reference `builder` and by the GPU `builder` CLI: the `.fmi` files must be identical, and the unmodified
    metaserver x4 + metaenumerate x5 must print the same mined substrings from either set.  Reduced to 12k reads
    per sample here; DSMFM_TEST_FULL_C2=1 runs the full 250k-read samples (minutes of CPU time)."""
    import dsmgen
    import mining
    full = bool(os.environ.get("DSMFM_TEST_FULL_C2"))
    exe = os.path.join(ROOT, "dsm-framework_b200", "builder")
    ours, theirs = {}, {}
    for i in range(1, 6):
        kw = dict(dsmgen.CONFIGS["C2-%d" % i])
        if not full:
            kw.update(n_reads=12_000, genome_len=12_000)
        name = "toydata-%d" % i
        for which, table in (("gpu", ours), ("ref", theirs)):
            d = tmp_path / which
            d.mkdir(exist_ok=True)
            fa = d / (name + ".fasta")
            dsmgen.fasta(**kw).tofile(str(fa))
            cmd = [exe, str(fa)] if which == "gpu" else [os.path.join(oracle.REF_DIR, "builder"), str(fa)]
            subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            table[name] = str(fa) + ".fmi"
        assert open(ours[name], "rb").read() == open(theirs[name], "rb").read(), name
    # --emax above log2(5): every mined substring is printed, whatever its entropy over the five samples
    got = mining.mine(ours, str(tmp_path / "mine_gpu"), emax="2.4")
    want = mining.mine(theirs, str(tmp_path / "mine_ref"), emax="2.4")
    assert sum(len(v) for v in want.values()) > 1000, "the mining run printed nothing"
    for h in want:
        assert hashlib.sha256(got[h]).hexdigest() == hashlib.sha256(want[h]).hexdigest(), "server %s output differs" % h
    # and with the mining CLIENT on the GPU as well: dsmfm_searcher_enumerate streams to the unmodified servers
    gpu = mining.mine(ours, str(tmp_path / "mine_gpu_client"), emax="2.4", client="gpu")
    for h in want:
        assert hashlib.sha256(gpu[h]).hexdigest() == hashlib.sha256(want[h]).hexdigest(), "server %s output differs (GPU client)" % h
