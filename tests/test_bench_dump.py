"""CPU suite: bench.py --dump-outputs writes the index a build hands its caller (dsmfm_index) as .npy files,
complete where it is small and as a fixed, seeded sample of the wavelet tree's bit vectors where it is not."""
import ctypes as C
import os

import numpy as np

import bench
import dsmfm


def _index(rng, nbits):
    """A dsmfm_index in host memory: root and one more internal node, three leaves (pre-order)."""
    keep, nodes = [], []
    for leaf, ch, nb in [(0, 65, nbits), (1, 65, 0), (0, 67, nbits // 2), (1, 67, 0), (1, 71, 0)]:
        nd = dsmfm.Node(leaf=leaf, ch=ch, nbits=nb, integers=0 if leaf else nb // 64 + 1)
        if not leaf:
            arrays = (rng.integers(0, 2**64, size=nd.integers, dtype=np.uint64),
                      np.cumsum(rng.integers(0, 257, size=nb // 256 + 1)).astype(np.uint64),
                      rng.integers(0, 256, size=nb // 64 + 1).astype(np.uint8))
            keep.append(arrays)
            nd.data, nd.Rs, nd.Rb = (a.ctypes.data_as(C.POINTER(t)) for a, t in zip(arrays, (C.c_uint64, C.c_uint64, C.c_uint8)))
        nodes.append(nd)
    table = (dsmfm.Node * len(nodes))(*nodes)
    idx = dsmfm.Index(n=nbits, samplerate=124, number_of_texts=7, max_text_length=9, n_nodes=len(nodes))
    idx.nodes = C.cast(table, C.POINTER(dsmfm.Node))
    idx.C[66] = 5
    idx.codetable[65] = dsmfm.Code(count=3, bits=2, code=1)
    return idx, keep, table


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_is_complete_below_the_sample_size(tmp_path):
    idx, keep, _ = _index(np.random.default_rng(1), 3000)
    bench.dump_outputs(str(tmp_path), idx)
    got = _load(str(tmp_path))
    assert sorted(got) == ["C", "codetable", "header", "nodes", "wt_rb", "wt_rs", "wt_words"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["header"].tolist() == [3000, 124, 7, 9, 5]
    assert got["C"][66] == 5 and got["codetable"][65].tolist() == [3, 2, 1]
    assert got["nodes"][:, 0].tolist() == [0, 1, 0, 1, 1] and got["nodes"][2, 2] == 1500
    w = got["wt_words"].astype(np.uint64)
    words = w[:, 0] | w[:, 1] << np.uint64(16) | w[:, 2] << np.uint64(32) | w[:, 3] << np.uint64(48)
    assert np.array_equal(words, np.concatenate([k[0] for k in keep]))
    assert np.array_equal(got["wt_rs"], np.concatenate([k[1] for k in keep]).astype(np.float64))
    assert np.array_equal(got["wt_rb"], np.concatenate([k[2] for k in keep]).astype(np.float32))


def test_dump_samples_the_same_entries_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 64)
    idx, keep, _ = _index(np.random.default_rng(2), 200_000)
    bench.dump_outputs(str(tmp_path / "a"), idx)
    bench.dump_outputs(str(tmp_path / "b"), idx)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert a["wt_words"].shape == (64, 4) and a["wt_rs"].shape == (64,) and a["wt_rb"].shape == (64,)
    rs = np.concatenate([k[1] for k in keep])
    assert np.isin(a["wt_rs"], rs.astype(np.float64)).all()
