"""`.sa` samples of the multi-GPU build: every rank derives its slice of the five sample vectors and writes its share
of `<prefix>.sa` (include/dsmfm.h, steps 8-11).  All ranks run on one GPU, one after the other
(multigpu.build_sharded_local), and through `builder --gpus N --samples`; the file must be the one the one-GPU build,
the oracle and the reference write."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
import oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
with open(os.path.join(GOLDEN, "manifest.json")) as _f:
    MANIFEST = json.load(_f)
EXE = os.path.join(ROOT, "dsm-framework_b200", "builder")


def _golden(name):
    with open(os.path.join(GOLDEN, name), "rb") as f:
        return f.read()


def _blocks(docs, world, device=None):
    import multigpu
    doc_list = bytes(docs).split(b"\0")[:-1]
    out = []
    for r in range(world):
        b, e = multigpu.block_of(len(doc_list), r, world)
        local = b"".join(d + b"\0" for d in doc_list[b:e])
        t = torch.frombuffer(bytearray(local), dtype=torch.uint8) if local else torch.empty(0, dtype=torch.uint8)
        out.append(t.cuda() if device == "cuda" and local else t)
    return out


def _build(blocks, rate, tmp_path, name, ranges=1, order=None):
    """-> (.fmi bytes, .sa bytes) written by the ranks (in `order`)"""
    import dsmfm
    import multigpu
    world = len(blocks)
    engines = [multigpu.CudaEngine(0, flags=dsmfm.FLAG_KEEP_SA, samplerate=rate) for _ in range(world)]
    sbs = multigpu.build_sharded_local(blocks, engines, ranges_per_gpu=ranges, samples=True)
    prefix = str(tmp_path / name)
    try:
        for r in (order or range(world)):
            sbs[r].write(prefix)
            sbs[r].write_samples(prefix)
    finally:
        for sb in sbs:
            sb.close()
    return _read(prefix + ".fmi"), _read(prefix + ".sa")


def _read(path):
    with open(path, "rb") as f:
        return f.read()


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("fn", sorted(MANIFEST["sa"]))
def test_ranks_write_the_golden_sa_files(fn, world, tmp_path):
    e = MANIFEST["sa"][fn]
    docs, _ = oracle.fasta_to_docs(_golden(e["case"] + ".fasta"))
    fmi, sa = _build(_blocks(docs, world), e["samplerate"], tmp_path, "g", ranges=1 + world % 2,
                     order=list(reversed(range(world))))
    assert sa == _golden(fn)
    assert fmi == oracle.fmi_from_docs(docs, e["samplerate"])


@pytest.mark.parametrize("world", [2, 4])
def test_ranks_reproduce_the_reference_digests(world, tmp_path):
    for key, e in sorted(MANIFEST["sa_digests"].items()):
        docs, _ = oracle.fasta_to_docs(cases.digest_cases()[e["case"]])
        _, sa = _build(_blocks(docs, world), e["samplerate"], tmp_path, key, ranges=2)
        assert len(sa) == e["bytes"] and hashlib.sha256(sa).hexdigest() == e["sha256"], key
    import dsmgen
    g = MANIFEST["generated"]["gen_20k"]
    fmi, sa = _build(_blocks(dsmgen.docs(**g["params"]).tobytes(), world), 0, tmp_path, "gen")
    assert hashlib.sha256(fmi).hexdigest() == g["fmi_sha256"]
    assert len(sa) == g["sa_bytes"] and hashlib.sha256(sa).hexdigest() == g["sa_sha256"]


def _random_docs(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "reads":
        docs, _ = oracle.fasta_to_docs(cases.rnd_fasta(seed, 1500, 100, minlen=20, genome=3000))
        return docs
    # sigma = 40: 8 bits per symbol
    parts = [bytes(rng.integers(33, 73, size=int(rng.integers(1, 80)), dtype=np.uint8)) for _ in range(500)]
    return b"".join(p + b"\0" for p in parts)


@pytest.mark.parametrize("world,ranges,lo_bits", [(2, 1, "12"), (3, 2, "14"), (5, 1, None)])
@pytest.mark.parametrize("kind", ["reads", "bytes"])
def test_random_collections_match_the_oracle(kind, world, ranges, lo_bits, tmp_path, monkeypatch):
    """DSMFM_POS_LO_BITS puts the high position bits into play; rate 1 samples every suffix, a rate above the longest
    document none (S = 0: empty `suffixes` and `suffixDocId`)."""
    if lo_bits:
        monkeypatch.setenv("DSMFM_POS_LO_BITS", lo_bits)
    docs = _random_docs(kind, world * 10 + ranges)
    longest = oracle.doc_stats(docs)[1]
    for rate in (1, 7, longest + 5):
        fmi, sa = _build(_blocks(docs, world, "cuda" if rate == 7 else None), rate, tmp_path, "r%d" % rate, ranges=ranges)
        assert sa == oracle.sa_file_from_docs(docs, rate), rate
        assert fmi == oracle.fmi_from_docs(docs, rate), rate


def test_ranks_without_documents_and_slices_without_samples(tmp_path):
    docs, _ = oracle.fasta_to_docs(cases.rnd_fasta(7, 5, 30))
    blocks = _blocks(docs, 8)  # five documents over eight ranks: three blocks hold nothing
    assert sum(b.numel() == 0 for b in blocks) == 3
    for rate in (1, 3, 64, 1000):
        fmi, sa = _build(blocks, rate, tmp_path, "s%d" % rate, order=[3, 7, 0, 5, 1, 6, 2, 4])
        assert sa == oracle.sa_file_from_docs(docs, rate), rate
        assert fmi == oracle.fmi_from_docs(docs, rate)


@pytest.mark.parametrize("rate", [64, 100])
def test_words_shared_by_many_ranks(rate, tmp_path):
    """World 8 over a few hundred symbols with 2 ranges per rank: every slice holds a handful of samples and end
    markers, so one word of `suffixDocId`, `Doc` and `suffixes` collects the bits of three ranks or more."""
    docs, _ = oracle.fasta_to_docs(cases.rnd_fasta(11, 12, 40, minlen=5))
    _, sa = _build(_blocks(docs, 8), rate, tmp_path, "w", ranges=2)
    assert sa == oracle.sa_file_from_docs(docs, rate)


def _doc_of(docs, sa):
    text = np.frombuffer(bytes(docs), dtype=np.uint8)
    starts = np.concatenate([[0], np.flatnonzero(text == 0)[:-1] + 1]).astype(np.uint64)
    sa = np.asarray(sa, dtype=np.uint64)
    doc = np.searchsorted(starts, sa, side="right") - 1
    return doc.astype(np.uint32), sa - starts[doc]


@pytest.mark.parametrize("rate", [1, 5, 40])
def test_searcher_locates_and_extracts_from_the_files_of_the_ranks(rate, tmp_path, monkeypatch):
    import dsmfm
    monkeypatch.setenv("DSMFM_POS_LO_BITS", "13")
    docs, nd = oracle.fasta_to_docs(cases.rnd_fasta(21, 900, 80, minlen=10, genome=2000))
    _build(_blocks(docs, 3), rate, tmp_path, "idx", ranges=2)
    _, sa = oracle.bwt(docs, want_sa=True)
    with dsmfm.Searcher(str(tmp_path / "idx.fmi")) as s:
        s.load_samples(str(tmp_path / "idx.sa"))
        doc, off = s.locate(np.arange(s.n, dtype=np.uint64))
        want_doc, want_off = _doc_of(docs, sa)
        assert np.array_equal(doc, want_doc) and np.array_equal(off, want_off)
        assert s.extract(np.arange(nd)) == bytes(docs).split(b"\0")[:-1]


@pytest.mark.parametrize("gpus", [2, 3, 8])
@pytest.mark.parametrize("name,rate", [("reads100", 16), ("small_random", 3), ("single", 3), ("mixed_alphabet", 16)])
def test_builder_cli_on_several_gpus_writes_the_samples(name, rate, gpus, tmp_path):
    fa = tmp_path / "in.fasta"
    fa.write_bytes(_golden(name + ".fasta"))
    r = subprocess.run([EXE, "--samples", "-s", str(rate), str(fa), str(tmp_path / "one")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([EXE, "--gpus", str(gpus), "--samples", "-s", str(rate), str(fa), str(tmp_path / "many")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = _read(str(tmp_path / "many.sa"))
    assert got == _read(str(tmp_path / "one.sa"))
    assert _read(str(tmp_path / "many.fmi")) == _read(str(tmp_path / "one.fmi"))
    golden = "%s.s%d.sa" % (name, rate)
    if golden in MANIFEST["sa"]:
        assert got == _golden(golden)


def test_builder_cli_on_several_gpus_writes_the_samples_of_an_empty_input(tmp_path):
    fa = tmp_path / "e.fasta"
    fa.write_bytes(b"")
    r = subprocess.run([EXE, "--gpus", "2", "--samples", str(fa)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert _read(str(fa) + ".sa") == oracle.sa_file_from_docs(b"", 124)
    r = subprocess.run([EXE, "--gpus", "2", "--host-parse", str(fa)], capture_output=True, text=True)
    assert r.returncode != 0 and "--host-parse" in r.stderr


def _two_builders(flags):
    """Two ranks through build_packed, by hand (-> builders, plan)"""
    import dsmfm
    blocks = [b"ACGTACGT\0TTGA\0", b"GGCA\0CAT\0A\0"]
    bs = [dsmfm.Builder(device=0, flags=flags, samplerate=2, shard_index=r, shard_count=2, shard_span=1) for r in range(2)]
    for b, blk in zip(bs, blocks):
        b.append_batch(blk)
    infos = [b.block_stats() for b in bs]
    plan = dsmfm.text_plan(infos)
    texts = [torch.zeros(int(plan.text_bytes), dtype=torch.uint8, device="cuda") for _ in bs]
    tops = [b.block_pack(plan, r, texts[r]) for r, b in enumerate(bs)]
    slot = int(plan.slot_words) * 8
    for r in range(2):
        texts[1 - r][r * slot:(r + 1) * slot].copy_(texts[r][r * slot:(r + 1) * slot])
    torch.cuda.synchronize()
    top = np.sum(np.stack(tops), axis=0, dtype=np.uint64)
    for b, t in zip(bs, texts):
        b.build_packed(plan, t, top)
    return bs, blocks


def test_calls_are_refused_without_the_flag_out_of_order_and_with_wrong_tables(tmp_path):
    import dsmfm
    bs, _ = _two_builders(0)
    try:
        with pytest.raises(dsmfm.DsmfmError) as e:
            bs[0].sa_slice_info()
        assert e.value.code == dsmfm.EINVAL
    finally:
        for b in bs:
            b.close()
    bs, blocks = _two_builders(dsmfm.FLAG_KEEP_SA)
    try:
        with pytest.raises(dsmfm.DsmfmError) as e:  # merge and write before the pieces
            bs[0].sa_pieces_merge(b"\0" * C.sizeof(dsmfm.PieceEdge) * dsmfm.SA_VECTORS * 2, 2)
        assert e.value.code == dsmfm.EINVAL
        with pytest.raises(dsmfm.DsmfmError):
            bs[0].sa_pieces_write(str(tmp_path / "x"), True)
        infos = [b.sa_slice_info() for b in bs]
        recs = [dsmfm.SaInfo.from_buffer_copy(i) for i in infos]
        assert sum(r.documents for r in recs) == 5 and sum(r.ends for r in recs) == 5
        assert [r.documents for r in recs] == [2, 3]
        for world in (1, 3):
            with pytest.raises(dsmfm.DsmfmError) as e:
                bs[0].sa_pieces_build(b"".join(infos[:1] * world), world, 0)
            assert e.value.code == dsmfm.EINVAL
        bad = dsmfm.SaInfo.from_buffer_copy(infos[1])
        bad.documents += 1
        with pytest.raises(dsmfm.DsmfmError) as e:  # does not add up to the collection
            bs[0].sa_pieces_build(infos[0] + bytes(bad), 2, 0)
        assert e.value.code == dsmfm.EINVAL and "documents" in str(e.value)
        with pytest.raises(dsmfm.DsmfmError):  # another builder's record
            bs[0].sa_pieces_build(infos[0] + infos[1], 2, 1)
        edges = [b.sa_pieces_build(b"".join(infos), 2, r) for r, b in enumerate(bs)]
        with pytest.raises(dsmfm.DsmfmError):
            bs[0].sa_pieces_build(b"".join(infos), 2, 0)
        with pytest.raises(dsmfm.DsmfmError):
            bs[0].sa_pieces_merge(b"".join(edges), 3)
        for b in bs:
            b.sa_pieces_merge(b"".join(edges), 2)
        for r in (1, 0):
            bs[r].sa_pieces_write(str(tmp_path / "hand"), r == 0)
        assert _read(str(tmp_path / "hand.sa")) == oracle.sa_file_from_docs(b"".join(blocks), 2)
    finally:
        for b in bs:
            b.close()


def test_struct_layout():
    import dsmfm
    assert C.sizeof(dsmfm.SaInfo) == 24
    assert [(n, getattr(dsmfm.SaInfo, n).offset) for n, _ in dsmfm.SaInfo._fields_] == [
        ("samples", 0), ("ends", 8), ("documents", 16)]
    assert C.sizeof(dsmfm.PieceEdge) == 96


def _ngpus():
    return torch.cuda.device_count()


def test_ranks_on_several_gpus_write_the_samples():
    if _ngpus() < 2:
        pytest.skip("needs 2 GPUs")
    port = 31500 + os.getpid() % 2000
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tests", "multigpu_samples_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MULTIGPU_SAMPLES_OK" in r.stdout
