"""Locate / extract throughput on the C3 workload (10 M reads of 100 bp, 2.02 G indexed symbols), one JSON line.

For each sample rate (124, the reference's default, and 16) the index is built with the suffix array kept, the samples
are attached from the in-memory `.sa` image, and the script times
  - locate_device on 2^24 random BWT positions (device arrays, so the kernel and not the copies is measured),
  - locate_ranges of the occurrences of 10^5 random 20-mers cut from the reads (host arrays in and out),
  - extract of 10^6 random documents (host arrays in and out),
each after warm-up, over repeated calls.  Every call ends in a synchronise of the searcher's stream: locate_device is
timed with CUDA events around the repeated calls (launch, synchronise and flag read-back included) and, in a separate
torch.profiler pass, by the device time of search_locate_kernel alone; the host-array calls are timed with a host clock
around the calls (copies in and out included).  Parity: 10^6 of the located positions
against the builder's suffix array, and every extracted document against the input.

    python tools_dev/locate_bench.py [--config C3] [--rates 124,16] [--repeat 10] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "dsm-framework_b200"))

import dsmfm  # noqa: E402
import dsmgen  # noqa: E402


def card():
    """name and power limit of GPU 0 (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # the numbers are still printed, marked as coming from an unnamed card
        return "unknown (%s)" % e, "unknown"


def mean_walk(doc_len, rate):
    """Mean LF steps of a locate at a uniformly random position of a document of doc_len symbols (+ terminator):
    the builder samples text positions e - rate + 1, e - 2 rate + 1, ... > s (e: terminator, s: first symbol), and a
    walk ends at a sampled position or at s."""
    s, e = 0, doc_len
    stop = np.zeros(e + 1, dtype=bool)
    stop[s] = True
    i = e - rate
    while i >= s:
        stop[i + 1] = True
        i -= rate
    last, total = 0, 0
    for x in range(e + 1):
        if stop[x]:
            last = x
        total += x - last
    return total / (e + 1)


def timed_events(fn, repeat, warmup=2):
    """seconds per call from CUDA events recorded before the first and after the last of `repeat` calls; each call
    synchronises the searcher's stream, so its launch, synchronise and flag read-back are inside the figure"""
    import torch
    for _ in range(warmup):
        fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(repeat):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / 1e3 / repeat


def kernel_ms(fn, name, calls=3):
    """mean device time of kernel `name` per call, from torch.profiler's CUDA activity in a pass of its own (None if the
    profiler reports no such kernel)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
    us = [getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
          for e in prof.key_averages() if name in e.key]
    return sum(us) / 1e3 / calls if us and sum(us) > 0 else None


def timed(fn, repeat, warmup=2):
    for _ in range(warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(repeat):
        fn()
    return (time.perf_counter() - t0) / repeat


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C3")
    ap.add_argument("--rates", default="124,16")
    ap.add_argument("--repeat", type=int, default=10)
    ap.add_argument("--positions", type=int, default=1 << 24)
    ap.add_argument("--patterns", type=int, default=100_000)
    ap.add_argument("--documents", type=int, default=1_000_000)
    ap.add_argument("--parity", type=int, default=1_000_000)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch

    cfg = dsmgen.CONFIGS[a.config]
    doc_size = 2 * cfg["read_len"] + 2  # complement + '-' + reverse + terminator
    docs = dsmgen.docs(**cfg)
    rows = docs.reshape(cfg["n_reads"], doc_size)
    rng = np.random.default_rng(2024)
    name, power = card()
    res = {"bench": "locate", "config": a.config, "card": name, "power_limit": power, "lib": os.path.basename(dsmfm.LIB_PATH),
           "positions": a.positions, "patterns": a.patterns, "documents": a.documents, "repeat": a.repeat, "rates": {}}
    parity = True
    for rate in [int(r) for r in a.rates.split(",")]:
        r = {}
        with dsmfm.Builder(device=0, flags=dsmfm.FLAG_KEEP_SA, samplerate=rate, expected_bytes=docs.size) as b:
            b.append_batch(docs)
            b.finish()
            img = b.sa_file()
            with dsmfm.Searcher(b) as s:
                n = s.n
                t0 = time.perf_counter()
                s.load_samples(img)
                r["attach_s"] = round(time.perf_counter() - t0, 3)
                r["sa_bytes"] = len(img)
                del img
                # 1. locate_device
                pos = torch.from_numpy(rng.integers(0, n, size=a.positions, dtype=np.int64)).cuda()
                doc = torch.empty(a.positions, dtype=torch.int32, device="cuda")
                off = torch.empty(a.positions, dtype=torch.int64, device="cuda")
                sec = timed_events(lambda: s.locate_device(pos, doc, off), a.repeat)
                r["locate_ms"] = round(sec * 1e3, 3)
                r["M_locates_per_s"] = round(a.positions / sec / 1e6, 2)
                kms = kernel_ms(lambda: s.locate_device(pos, doc, off), "search_locate_kernel")
                r["locate_kernel_ms"] = None if kms is None else round(kms, 3)
                r["M_locates_per_s_kernel"] = None if kms is None else round(a.positions / kms / 1e3, 2)
                r["mean_walk_model"] = round(mean_walk(doc_size - 1, rate), 2)
                # parity of the first `parity` located positions against the suffix array, gathered chunk by chunk
                m = min(a.parity, a.positions)
                qp = pos[:m].cpu().numpy()
                got_doc = doc[:m].cpu().numpy().view(np.uint32)
                got_off = off[:m].cpu().numpy().astype(np.uint64)
                order = np.argsort(qp)
                want = np.empty(m, dtype=np.uint64)
                chunk = 1 << 28
                for first in range(0, n, chunk):
                    lo, hi = np.searchsorted(qp[order], [first, min(first + chunk, n)])
                    if lo == hi:
                        continue
                    sa = b.suffix_array(first, min(chunk, n - first))
                    want[order[lo:hi]] = sa[qp[order[lo:hi]] - first]
                ok = np.array_equal(got_doc, (want // doc_size).astype(np.uint32)) and np.array_equal(got_off, want % doc_size)
                r["parity_locate"] = bool(ok)
                parity &= bool(ok)
                del pos, doc, off
                # 2. locate_ranges of 20-mers cut from the reads
                ks = rng.integers(0, cfg["n_reads"], size=a.patterns)
                at = rng.integers(0, doc_size - 1 - 20, size=a.patterns)
                pats = [rows[k, o:o + 20].tobytes() for k, o in zip(ks, at)]
                sp, ep = s.count(pats)
                out = {}

                def ranges():
                    out["r"] = s.locate_ranges(sp, ep)
                sec = timed(ranges, a.repeat)
                occ = int(out["r"][2][-1])
                r["occurrences"] = occ
                r["locate_ranges_ms"] = round(sec * 1e3, 3)
                r["M_occurrences_per_s"] = round(occ / sec / 1e6, 2)
                # every occurrence of a pattern cut from read k at offset o: read k's own is among them
                d, o, st = out["r"]
                mine = [np.any((d[st[j]:st[j + 1]] == ks[j]) & (o[st[j]:st[j + 1]] == at[j])) for j in range(min(a.patterns, 20000))]
                r["parity_ranges"] = bool(all(mine))
                parity &= r["parity_ranges"]
                # 3. extract of random documents (the raw entry point: no Python objects per document)
                kd = np.ascontiguousarray(rng.integers(0, cfg["n_reads"], size=a.documents).astype(np.uint32))
                offs = np.empty(a.documents + 1, dtype=np.uint64)
                buf = np.empty(a.documents * (doc_size - 1), dtype=np.uint8)
                L = dsmfm.lib()

                def extract():
                    rc = L.dsmfm_searcher_extract(s._h, kd.ctypes.data, kd.size, buf.ctypes.data, buf.size, offs.ctypes.data)
                    if rc != dsmfm.OK:
                        raise dsmfm.DsmfmError(rc, L.dsmfm_searcher_last_error(s._h).decode())
                sec = timed(extract, a.repeat)
                r["extract_ms"] = round(sec * 1e3, 3)
                r["M_documents_per_s"] = round(a.documents / sec / 1e6, 3)
                ok = np.array_equal(buf.reshape(a.documents, doc_size - 1), rows[kd, :doc_size - 1])
                r["parity_extract"] = bool(ok)
                parity &= bool(ok)
        res["n"] = int(n)
        res["rates"][str(rate)] = r
    res["parity"] = bool(parity)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if parity else 1


if __name__ == "__main__":
    sys.exit(main())
