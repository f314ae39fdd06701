#!/usr/bin/env python
"""bench.py -- FM-index build throughput (Mbp/s) of the B200-native `builder` path.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU implementation
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also writes the index of the last timed step

A step = one complete FM-index build (pack, suffix sort, BWT, HuffWT + BitRank) of one synthetic
sample.  N=1: the 1 Gbp sample of BASELINE.json configs[2] (SURVEY 8d "C3": 10M x 100-bp reads,
n = 2.02 G indexed symbols).  N>1 (torchrun, one rank per GPU): every rank holds its own 1 Gbp block
of reads and the N GPUs build ONE index of the N Gbp collection (weak scaling; BASELINE.json
configs[3] shape): NCCL all-gather of the raw text, key-range sharded suffix sort (every GPU sorts
its share of the global suffix order from the replicated text), BWT slices sent to rank 0, which
builds the wavelet tree (dsm-framework_b200/multigpu.py).

value   = input bases of all ranks / max-over-ranks device time, documents already resident in HBM.
e2e     = the same through the C ABI with HOST buffers: dsmfm_append_batch from pinned host memory
          (H2D inside the timed region) ... dsmfm_finish (sections copied back to the host).
roofline: the dominant kernel is the one-sweep LSD radix pass (6 passes, each one launch per portion of
          <= 2^29 pairs: 24 launches per 1 Gbp build); achieved = 24 B/pair (8+4 read, 8+4 written) x
          pairs of a launch / mean launch time (CUDA events on the build stream, recorded inside the
          library around the passes of every timed step, divided by the number of launches).
cpu_baseline: the UNMODIFIED reference `builder` (oracle/_ref/builder, single-threaded as shipped)
          on a bounded toydata-shaped sample, on this box's host cores, rank 0 at N=1 only.
fasta_e2e (N=1): the path of the drop-in CLI -- FASTA bytes in pinned host memory, parsed and transformed on the GPU
          (dsmfm_append_fasta), sections copied back; same workload, same unit.
search (N=1): dsmfm_searcher_lf_device on the index of the workload, G LF queries/s (the query half of the index).
roofline_refine: the refinement phase (second largest share of the step) against the same HBM peak.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "dsm-framework_b200"))

WORKLOADS = {
    # name -> generator parameters (dsmgen.CONFIGS) ; per-rank seed offset is added for N>1
    "C3": "C3",
    "C1": "C1",
    "C5": "C5",  # high repetition: 4 genomes at 200x coverage, error free (BASELINE.json configs[4])
    "C4": "C4",  # 16 Gbp metagenome: 2000 x 1 Mbp genomes at 8x (BASELINE.json configs[3]; with --reads and --shared-genomes)
}
CPU_SAMPLE = dict(seed=1, pool_seed=1, pool_size=10, n_genomes=10, genome_len=100_000, n_reads=100_000,
                  read_len=100, sub=0.005, pn=0.001)  # 10 Mbp at the 10x coverage of C1


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed loop (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--reads", type=int, default=0, help="override the number of reads (debugging)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the FASTA front-end and query-side measurements (N=1)")
    ap.add_argument("--ranges-per-gpu", type=int, default=1, help="N>1: key ranges sorted one after the other per GPU")
    ap.add_argument("--no-full-parity", action="store_true", help="N>1: skip the one-GPU rebuild of the full collection (parity)")
    ap.add_argument("--full-parity", action="store_true",
                    help="N>4: rebuild the full collection on one GPU as well (minutes of host time at 8 x 1 Gbp; default only up to N=4)")
    ap.add_argument("--shared-genomes", action="store_true",
                    help="N>1: all ranks draw their reads from the SAME genomes (strong-scaling shape of C4 / C5: --reads = total / N)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="one GPU: write the index the last timed step built to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU build computed (--impl ours)")
    return args


class ClockSampler:
    """SM clocks / throttle reasons / power DURING the timed region (B200_PROFILING.md's clocks line).

    The counters are the ones `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.*` prints,
    read through NVML from a thread of this process every 100 ms (more samples per timed region than a child process
    polling every 250 ms, and nothing else competing for the driver).  An `nvidia-smi -lms 250` child process is the
    fallback when pynvml is missing; BENCH_CLOCKS=smi selects it.  (In one run the steps that coincided with a sample
    of the child process were 10 ms longer, profiles/r2c_bench_1gpu_smi.json; a repeat showed no such effect.)"""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, pci_bus_id=None):
        self.index = index
        self.pci_bus_id = pci_bus_id
        self.proc = None
        self.thread = None
        self.nvml = None
        self.stop_flag = threading.Event()
        self.lines = []      # nvidia-smi csv lines
        self.samples = []    # (sm_mhz, max_mhz, watts, reason names)
        self.source = None

    def start(self):
        if os.environ.get("BENCH_CLOCKS", "nvml") != "smi":
            try:
                import pynvml
                pynvml.nvmlInit()
                handle = None
                if self.pci_bus_id:
                    try:
                        handle = pynvml.nvmlDeviceGetHandleByPciBusId(self.pci_bus_id.encode())
                    except Exception:
                        handle = None
                if handle is None:
                    handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
                self.nvml, self.handle, self.source = pynvml, handle, "nvml"
                self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
                self.thread = threading.Thread(target=self._poll, daemon=True)
                self.thread.start()
                return
            except Exception:
                self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "250"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 250"
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.handle
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"), (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"), (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        while True:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                watts = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.samples.append((sm, self.max_mhz, watts, [nm for bit, nm in bits if mask & bit]))
            except Exception:
                pass
            if self.stop_flag.wait(0.1):
                return

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=5)
        elif self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            for ln in self.lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 7:
                    continue
                try:
                    self.samples.append((float(f[0]), float(f[1]), float(f[2]),
                                         [nm for nm, v in zip(self.NAMES, f[3:7]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"]}
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "source": self.source}
        reasons = set()
        for smp in self.samples:
            reasons.update(smp[3])
        # median over the samples taken under load (the upper half by power draw)
        under_load = sorted(self.samples, key=lambda x: x[2])[len(self.samples) // 2:]
        load = sorted(x[0] for x in under_load)
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(x[1] for x in self.samples), "reasons": sorted(reasons),
                "samples": len(self.samples), "power_w_max": round(max(x[2] for x in self.samples), 2), "source": self.source}


def section_bytes(idx):
    total = 0
    for i in range(idx.n_nodes):
        nd = idx.nodes[i]
        if not nd.leaf:
            total += 8 * nd.integers + 8 * (nd.nbits // 256 + 1) + (nd.nbits // 64 + 1)
    return total


def fmi_sha256(index, dsmfm):
    """SHA-256 of the `.fmi` bytes FMIndex::save would write for these sections (dsmfm_fmi_serialize)."""
    import hashlib
    blob = dsmfm.fmi_bytes(index)
    return hashlib.sha256(blob).hexdigest(), len(blob)


def reference_digest(workload, kw):
    """Digest of the `.fmi` the UNMODIFIED reference wrote for exactly these generator parameters
    (tests/golden/fullsize.json, made by tests/golden/make_fullsize_golden.py), or None."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "fullsize.json")) as f:
            table = json.load(f)
    except Exception:
        return None
    for name, rec in table.items():
        if all(rec["params"].get(k) == v for k, v in kw.items()) and len(rec["params"]) == len(kw):
            return dict(rec, name=name)
    return None


def sha256_file(path):
    import hashlib
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            blk = f.read(1 << 24)
            if not blk:
                break
            h.update(blk)
    return h.hexdigest(), os.path.getsize(path)


DUMP_SAMPLE = 1 << 20  # entries sampled from each of the three bit-vector arrays of the wavelet tree


def dump_outputs(out_dir, idx):
    """--dump-outputs: the index as dsmfm_fetch hands it to a caller, written to <out_dir>/<name>.npy so that two builds
    of the project can be compared array for array.  header (n, samplerate, number_of_texts, max_text_length, n_nodes),
    C, codetable (count, bits, code per symbol) and nodes (leaf, ch, nbits, integers per node, pre-order) are complete,
    in float64.  The wavelet tree's bit vectors (about 0.8 GB at C3) are sampled: DUMP_SAMPLE positions drawn with a
    fixed seed over each array of the internal nodes concatenated in pre-order -- wt_words (64-bit words as four 16-bit
    parts, low first, float32), wt_rs (superblock ranks, float64), wt_rb (block ranks, float32).  About 30 MB in all."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def save(name, arr):
        np.save(os.path.join(out_dir, name + ".npy"), arr)

    nodes = [idx.nodes[i] for i in range(idx.n_nodes)]
    save("header", np.array([idx.n, idx.samplerate, idx.number_of_texts, idx.max_text_length, idx.n_nodes], dtype=np.float64))
    save("C", np.array(idx.C[:], dtype=np.float64))
    save("codetable", np.array([(c.count, c.bits, c.code) for c in idx.codetable], dtype=np.float64).reshape(-1, 3))
    save("nodes", np.array([(nd.leaf, nd.ch, nd.nbits, nd.integers) for nd in nodes], dtype=np.float64).reshape(-1, 4))

    inner = [nd for nd in nodes if not nd.leaf]

    def sample(field, length, dtype, seed):
        sizes = [length(nd) for nd in inner]
        off = np.concatenate([[0], np.cumsum(sizes, dtype=np.int64)])
        total = int(off[-1])
        rng = np.random.default_rng(seed)
        pos = np.sort(rng.integers(0, total, size=DUMP_SAMPLE)) if total > DUMP_SAMPLE else np.arange(total)
        which = np.searchsorted(off, pos, side="right") - 1
        out = np.empty(pos.size, dtype=dtype)
        for j, nd in enumerate(inner):
            sel = which == j
            if sel.any():
                out[sel] = np.ctypeslib.as_array(getattr(nd, field), shape=(sizes[j],))[pos[sel] - off[j]]
        return out

    words = sample("data", lambda nd: nd.integers, np.uint64, 1)
    save("wt_words", ((words[:, None] >> np.arange(0, 64, 16, dtype=np.uint64)) & np.uint64(0xFFFF)).astype(np.float32))
    save("wt_rs", sample("Rs", lambda nd: nd.nbits // 256 + 1, np.uint64, 2).astype(np.float64))
    save("wt_rb", sample("Rb", lambda nd: nd.nbits // 64 + 1, np.uint8, 3).astype(np.float32))


def multi_gpu_parity(args, dist, torch, dsmfm, dsmgen, multigpu, engine, host_docs, kw, rank, world, local):
    """Parity of the N-GPU build (outside the timed regions).
    (1) preflight at reduced size: 100k reads per rank built by the N ranks, every rank writing its share of the
        file, against the SAME documents built unsharded on one GPU (the path pinned to the reference's digests);
    (2) full size: the index of the workload just timed, written by the N ranks, against a one-GPU build of the
        same N x 1 Gbp collection on rank 0 (key ranges sorted one after the other; --no-full-parity skips it)."""
    import shutil
    import tempfile
    import traceback
    box = [tempfile.mkdtemp(prefix="dsmfm_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None) if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    tmp = box[0]
    out = {"world": world}
    try:
        # ---- (1) reduced size ----
        small = dict(kw, n_reads=100_000, genome_len=max(10_000, kw["genome_len"] // 100))
        pool_step = 0 if args.shared_genomes else 1000
        kws = [dict(small, seed=small["seed"] - 1000 * rank + 1000 * r, pool_seed=small["pool_seed"] - pool_step * rank + pool_step * r)
               for r in range(world)]
        mine = torch.from_numpy(dsmgen.docs(**kws[rank])).pin_memory()
        sb = multigpu.build_sharded(dist, mine, engine, ranges_per_gpu=args.ranges_per_gpu)
        sb.write(os.path.join(tmp, "small"))
        sb.close()
        dist.barrier()
        if rank == 0:
            got, size = sha256_file(os.path.join(tmp, "small.fmi"))
            with dsmfm.Builder(device=local) as b1:
                for r in range(world):
                    b1.append_batch(dsmgen.docs(**kws[r]))
                want, wsize = fmi_sha256(b1.finish(), dsmfm)
            out["preflight"] = {"reads_per_rank": small["n_reads"], "sha256": got, "fmi_bytes": size,
                                "matches": bool(got == want and size == wsize),
                                "against": "the same documents built unsharded on one GPU (dsmfm_finish)"}
        # ---- (2) the workload itself ----
        sb = multigpu.build_sharded(dist, host_docs, engine, ranges_per_gpu=args.ranges_per_gpu)
        sb.write(os.path.join(tmp, "full"))
        sb.close()
        dist.barrier()
        if rank == 0:
            got, size = sha256_file(os.path.join(tmp, "full.fmi"))
            out.update({"sha256": got, "fmi_bytes": size, "matches": None, "against": None})
            os.remove(os.path.join(tmp, "full.fmi"))
            if not args.no_full_parity and (world <= 4 or args.full_parity):
                try:
                    dsmfm.lib().dsmfm_release_cached(local)
                    torch.cuda.empty_cache()
                    k = max(2, world)
                    with dsmfm.Builder(device=local, shard_index=0, shard_count=k, shard_span=k) as b1:
                        for r in range(world):
                            kr = dict(kw, seed=kw["seed"] - 1000 * rank + 1000 * r, pool_seed=kw["pool_seed"] - pool_step * rank + pool_step * r)
                            b1.append_batch(host_docs if r == rank else dsmgen.docs(**kr))
                        b1.build_device()
                        info = b1.shard_info()
                        b1.assemble(int(info.bwt_dev), int(info.n_total))
                        want, wsize = fmi_sha256(b1.fetch(), dsmfm)
                    out["matches"] = bool(got == want and size == wsize)
                    out["against"] = ("the same %d x %.2f Gbp collection built on ONE GPU (rank 0: %d key ranges sorted one after "
                                      "the other, wavelet tree over the whole BWT), itself pinned to the reference by the C3 digest "
                                      "at N=1" % (world, kw["n_reads"] * kw["read_len"] / 1e9, k))
                except Exception as e:  # (e.g. not enough memory for the one-GPU build): the preflight still stands
                    out["full_size_error"] = "%s: %s" % (type(e).__name__, str(e)[:300])
                    traceback.print_exc(file=sys.stderr)
                    out["matches"] = out.get("preflight", {}).get("matches")
                    out["against"] = "preflight only (the one-GPU build of the full collection failed, see full_size_error)"
            else:
                out["matches"] = out.get("preflight", {}).get("matches")
                out["against"] = ("preflight only: the one-GPU rebuild of the full collection is run up to N=4 by default "
                                  "(--full-parity forces it), where it matched; the full-size file's digest is `sha256`")
            if out.get("preflight", {}).get("matches") is False:
                out["matches"] = False
        dist.barrier()
    finally:
        if rank == 0:
            shutil.rmtree(tmp, ignore_errors=True)
    return out if rank == 0 else None


def cpu_reference_run(threads, params, tmpdir):
    """Times the reference's own CPU implementation on a bounded sample.  threads == 1: the stock
    `builder` binary; threads > 1: oracle/_ref/ref_driver, which drives the same reference classes
    with incbwt's OpenMP sort enabled (RLCSABuilder's `threads` argument)."""
    import dsmgen
    ref = os.path.join(ROOT, "oracle", "_ref")
    bases = params["n_reads"] * params["read_len"]
    if threads <= 1:
        path = os.path.join(tmpdir, "cpu_sample.fasta")
        dsmgen.fasta(**params).tofile(path)
        t0 = time.perf_counter()
        subprocess.run([os.path.join(ref, "builder"), path], check=True, stdout=subprocess.DEVNULL,
                       stderr=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
    else:
        path = os.path.join(tmpdir, "cpu_sample.docs")
        dsmgen.docs(**params).tofile(path)
        env = dict(os.environ, OMP_NUM_THREADS=str(threads))
        t0 = time.perf_counter()
        subprocess.run([os.path.join(ref, "ref_driver"), "fmi", path, os.path.join(tmpdir, "cpu_sample"),
                        str(threads)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
        dt = time.perf_counter() - t0
    return bases / dt / 1e6, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import tempfile
    have = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_driver"))
    if not have:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref was not built (needs /root/reference at build time)"}))
        return 0
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, 64))
    times = []
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(args.warmup + args.steps):
            mbps, dt = cpu_reference_run(threads, CPU_SAMPLE, tmp)
            if i >= args.warmup:
                times.append(dt)
    bases = CPU_SAMPLE["n_reads"] * CPU_SAMPLE["read_len"]
    total = sum(times)
    value = bases * len(times) / total / 1e6
    sample = ("%d x %d-bp reads (%.0f Mbp, 10x coverage, sub 0.005, N 0.001) per step; the reference classes "
              "(RLCSABuilder -> FMIndex -> HuffWT) driven by oracle/ref_driver.cpp with incbwt's OpenMP sort on "
              "%d threads; the documents are handed over ready-made (FASTA parsing and transform() are NOT timed, "
              "which favours the CPU arm; a single 512 MiB batch, so incbwt's merge by backward search never runs)"
              % (CPU_SAMPLE["n_reads"], CPU_SAMPLE["read_len"], bases / 1e6, threads))
    line = {"impl": "reference", "metric": "fm_index_build_throughput", "value": round(value, 4), "unit": "Mbp/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1000 * total / len(times), 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "bounded sample of " + args.workload + ": " + sample},
            "cpu_baseline": {"value": round(value, 4), "unit": "Mbp/s", "cores": threads, "kind": "reference",
                             "sample": sample},
            "e2e": {"value": round(value, 4), "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def fasta_front_end(args, kw, local, stream, torch, dsmfm, dsmgen):
    """The path of the drop-in CLI: FASTA bytes in pinned host memory -> dsmfm_append_fasta (record loop, normalize and
    transform on the GPU) -> dsmfm_finish (sections in host memory).  Same workload, same metric."""
    import numpy as np
    fa = dsmgen.fasta(**kw)
    host = torch.empty(fa.size, dtype=torch.uint8, pin_memory=True)
    host.numpy()[:] = fa
    del fa
    bases = kw["n_reads"] * kw["read_len"]

    def step():
        b = dsmfm.Builder(device=local, stream=stream.cuda_stream)
        info = b.append_fasta(host)
        b.finish()
        s = b.stats()
        b.close()
        return info, s

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        info, s = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    return {"value": round(bases / dt / 1e6, 2), "unit": "Mbp/s", "ms_per_step": round(1000 * dt, 2),
            "fasta_bytes_per_step": int(host.numel()), "documents": int(info["documents"]),
            "api": "dsmfm_create / dsmfm_append_fasta (pinned host buffer, parsed on the GPU) / dsmfm_finish / dsmfm_destroy",
            "gpu_launches_per_step": int(s.kernel_launches), "build_device_ms": round(s.ms_total, 2),
            "build_wall_ms": round(s.ms_wall_build, 2), "alloc_wall_ms": round(s.ms_wall_alloc, 2),
            "fetch_wall_ms": round(s.ms_wall_fetch, 2)}


def query_side(host_docs, local, stream, torch, dsmfm, reps):
    """dsmfm_searcher_lf_device on the index of the workload: random (symbol, position) LF queries, device arrays,
    CUDA events.  Every query walks the Huffman code of its symbol: per level one 8-byte Rs, one 1-byte Rb and one
    8-byte bit word, each a random access to HBM."""
    b = dsmfm.Builder(device=local, stream=stream.cuda_stream)
    b.append_batch(host_docs)
    b.finish()
    s = dsmfm.Searcher(b, device=local)
    n = s.n
    b.close()
    m = 1 << 26
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    qi = torch.randint(0, n, (m,), dtype=torch.int64, device="cuda", generator=g)
    qc = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")[torch.randint(0, 4, (m,), device="cuda", generator=g)]
    out = torch.empty(m, dtype=torch.int64, device="cuda")
    for _ in range(2):
        s.lf_device(qc, qi, out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        s.lf_device(qc, qi, out)  # runs on the searcher's stream and waits for it
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    s.close()
    return {"value": round(m / ms / 1e6, 3), "unit": "G LF queries/s", "queries_per_launch": m, "ms_per_launch": round(ms, 3),
            "index_symbols": int(n), "api": "dsmfm_searcher_lf_device (FMIndex::LF over HuffWT::rank, one thread per query)"}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    # ONE JSON line on stdout and nothing else: whatever a library prints to file descriptor 1 (NCCL's version
    # banner, for one) goes to stderr; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs is for a one-GPU run")
    if world > 1:  # torchrun pins OMP_NUM_THREADS to 1; the read generator (input preparation) is OpenMP code
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // world))
    import torch
    import dsmfm
    import dsmgen

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this path has no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's banner / debug lines off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    kw = dict(dsmgen.CONFIGS[WORKLOADS[args.workload]])
    kw["seed"] += 1000 * rank  # every rank holds its own block of reads, drawn from its own genomes
    pool_step = 0 if args.shared_genomes else 1000
    kw["pool_seed"] += pool_step * rank  # (coverage stays that of the workload as N grows, like C4 vs C3)
    if args.reads:
        kw["n_reads"] = args.reads
    n_reads, L = kw["n_reads"], kw["read_len"]
    bases = n_reads * L
    nbytes = n_reads * (2 * L + 2)

    host_docs = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dsmgen.docs(out=host_docs, **kw)
    dev_docs = host_docs.cuda(non_blocking=False)
    stream = torch.cuda.current_stream()
    flags = 0
    last_build = [None]

    if world > 1:
        import multigpu
        engine = multigpu.CudaEngine(local, flags=flags)
        launches = [0]

        def sharded(docs, fetch=True):
            sb = multigpu.build_sharded(dist, docs, engine, ranges_per_gpu=args.ranges_per_gpu, fetch=fetch)
            s, out_bytes = sb.build_stats(), sb.section_bytes
            sb.close()
            launches[0] += s.kernel_launches
            return s, out_bytes

        def device_step(last=False):  # inputs resident in HBM, every rank's share of the sections left in its HBM
            return sharded(dev_docs, False)[0]

        def e2e_step():
            return sharded(host_docs)
    else:
        def device_step(last=False):
            b = dsmfm.Builder(device=local, stream=stream.cuda_stream, expected_bytes=nbytes, flags=flags)
            b.append_batch_device(dev_docs)
            b.build_device()
            s = b.stats()
            if last and args.dump_outputs:
                last_build[0] = b  # its sections stay in HBM until they are dumped behind the timed region
            else:
                b.close()
            return s

        def e2e_step():
            b = dsmfm.Builder(device=local, stream=stream.cuda_stream, expected_bytes=nbytes, flags=flags)
            b.append_batch(host_docs)
            idx = b.finish()
            out_bytes = section_bytes(idx)
            s = b.stats()
            b.close()
            return s, out_bytes

    # ---- device-resident throughput ("value") ------------------------------------------------------
    for _ in range(args.warmup):
        device_step()
    try:  # the NVML handle by PCI address: NVML's indices need not be CUDA's
        pr = torch.cuda.get_device_properties(local)
        pci = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        pci = None
    sampler = ClockSampler(local, pci)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    stats, step_wall = [], []
    for i in range(args.steps):
        t_s = time.perf_counter()
        stats.append(device_step(last=i == args.steps - 1))
        step_wall.append(round(1000 * (time.perf_counter() - t_s), 1))
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    if last_build[0] is not None:
        dump_outputs(args.dump_outputs, last_build[0].fetch())
        last_build[0].close()

    # ---- end to end through the C ABI with host buffers ("e2e") ---------------------------------------
    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_out = [e2e_step() for _ in range(args.steps)]
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], device="cuda")
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    barrier()
    t_e2e = float(t_e2e.item())
    n_launch = torch.tensor([sum(s.kernel_launches for s in stats), e2e_out[-1][1]], dtype=torch.int64, device="cuda")
    if dist is not None:
        dist.all_reduce(n_launch)
    n_launch, d2h_bytes = int(n_launch[0].item()), int(n_launch[1].item())
    parity = multi_gpu_parity(args, dist, torch, dsmfm, dsmgen, multigpu, engine, host_docs, kw, rank, world, local) if world > 1 else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650 GB/s (of fallback)"
    s0 = stats[-1]
    pass_ms = sum(s.ms_sort_pass for s in stats) / len(stats)
    achieved = s0.sort_pass_bytes / (pass_ms * 1e-3) / 1e9 if pass_ms > 0 else 0.0
    profile = {}
    try:
        profile = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    except Exception:
        pass

    line = {
        "metric": "fm_index_build_throughput",
        "value": round(world * bases * args.steps / (ms_total * 1e-3) / 1e6, 2),
        "unit": "Mbp/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(ms_total / args.steps, 3),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic",
        "config": {
            "workload": "%s: %d x %d-bp ACGTN reads per GPU (%.2f Gbp, n = %d indexed symbols): every section of the .fmi "
                        "(suffix sort -> BWT -> C[] -> HuffWT -> BitRank).  The headline build sorts the suffixes only as far "
                        "as the BWT needs (tie groups whose members share one BWT symbol stay unsorted: the .fmi holds no "
                        "suffix array); the build that finishes the whole suffix array is `with_suffix_array`"
                        % (args.workload, n_reads, L, bases / 1e9, nbytes),
            "parallelism": "1 GPU" if world == 1 else
                           "%d GPUs build ONE index of %.2f Gbp: every rank packs its block, NCCL all-gather of the PACKED slots "
                           "(3 bits per symbol), key-range sharded suffix sort from the replicated packed text (%d range(s) per "
                           "GPU, no exchange during the sort), every rank builds its share of the wavelet tree and BitRank "
                           "directories on its own GPU and copies it to its own host (no funnel through one GPU)"
                           % (world, world * bases / 1e9, args.ranges_per_gpu),
            "cache": "inputs (%.2f GB) and sort buffers are far larger than the 126 MB L2; no flush needed" % (nbytes / 1e9),
            "bits_per_symbol": s0.bits_per_symbol,
            "refine_rounds": s0.rounds,
            "active_fraction_per_round": [round(s0.active[r] / s0.n, 4) for r in range(min(s0.rounds, 32))],
            "phase_ms": {"pack": round(s0.ms_pack, 2), "sort": round(s0.ms_sort, 2), "refine": round(s0.ms_refine, 2),
                         "bwt": round(s0.ms_bwt, 2), "wavelet": round(s0.ms_wt, 2), "total": round(s0.ms_total, 2)},
            "device_bytes_peak": s0.device_bytes_peak,
            "step_wall_ms": step_wall,
            "step_device_ms": [round(s.ms_total, 1) for s in stats],
            "step_build_wall_ms": [round(s.ms_wall_build, 1) for s in stats],
            "step_alloc_wall_ms": [round(s.ms_wall_alloc, 1) for s in stats],
        },
        "clocks": clocks,
        "e2e": {
            "value": round(world * bases * args.steps / t_e2e / 1e6, 2),
            "unit": "Mbp/s",
            "h2d_bytes_per_step": world * nbytes,
            "d2h_bytes_per_step": d2h_bytes,
            "ms_per_step": round(1000 * t_e2e / args.steps, 2),
            "api": "dsmfm_create / dsmfm_append_batch (pinned host buffer) / dsmfm_finish / dsmfm_destroy" if world == 1 else
                   "per rank: dsmfm_create / dsmfm_append_batch (pinned host buffer) / dsmfm_block_stats / dsmfm_block_pack / "
                   "NCCL all-gather of the packed slots / dsmfm_build_packed / dsmfm_pieces_build (the rank's share of the sections "
                   "copied to ITS host memory) / dsmfm_pieces_merge / dsmfm_destroy",
        },
        "gpu_launches": n_launch,
        "roofline": {
            "bound": "hbm",
            "kernel": "onesweep_kernel: one launch of the LSD radix sort over (u64 key, u32 suffix) pairs; %d passes x %d "
                      "portion(s) of <= 2^29 pairs = %d launches per build" % (
                          s0.sort_passes, max(1, s0.sort_launches // max(1, s0.sort_passes)), s0.sort_launches),
            "achieved": round(achieved, 1),
            "peak": peak,
            "unit": "GB/s",
            "frac": round(achieved / peak, 4),
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": s0.sort_pass_bytes,
            "ms_per_launch": round(pass_ms, 4),
            "traffic": profile.get("onesweep_dram_bytes_per_launch"),
            "traffic_note": profile.get("note"),
        },
    }

    # Second kernel of the step: the refinement.  Only the tie groups whose members carry different BWT symbols are
    # sorted (BWT-only build); its algorithmic bytes: per member 4+1 B read and 1 B written back (suffix, BWT symbol),
    # 8 B per key gathered from the packed text, and the two bitmaps (group heads, symbol differences) of n/8 B each.
    members = s0.refine_members
    ref_bytes = 6 * members + 8 * s0.refine_key_fetches + s0.n // 4
    ref_ms = sum(s.ms_refine for s in stats) / len(stats)
    ref_ach = ref_bytes / (ref_ms * 1e-3) / 1e9 if ref_ms > 0 else 0.0
    line["roofline_refine"] = {
        "bound": "hbm", "kernel": "refinement phase: mark/count/compact the groups with mixed BWT symbols, refine_warps_kernel "
                                  "(%d launch(es); every warp resolves the groups of its part of a 1024-slot window in shared "
                                  "memory, keys gathered from the packed text), scatter the BWT bytes back" % s0.refine_launches,
        "achieved": round(ref_ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ref_ach / peak, 4),
        "algorithmic_bytes": ref_bytes, "ms": round(ref_ms, 3),
        "tie_group_members": int(sum(s0.active[r] for r in range(min(s0.rounds, 1)))), "members_sorted": int(members),
        "keys_gathered": s0.refine_key_fetches, "traffic": profile.get("refine_dram_bytes_per_launch"),
        "traffic_note": profile.get("refine_note"),
        "note": "random 16-byte gathers: the bound is DRAM row activations (about 56 G accesses/s measured, "
                "tools_dev/gather_bench.cu), not bytes"}

    if parity is not None:
        line["parity"] = parity
    if world == 1:
        # the same workload with the WHOLE suffix array finished (DSMFM_FLAG_KEEP_SA: what BASELINE.json's "SA" and the
        # .sa sampling need); device-resident inputs, CUDA events on the build stream like `value`
        sa_steps = args.steps
        sa_stats = []
        for i in range(1 + sa_steps):
            b = dsmfm.Builder(device=local, stream=stream.cuda_stream, expected_bytes=nbytes, flags=dsmfm.FLAG_KEEP_SA)
            b.append_batch_device(dev_docs)
            b.build_device()
            if i:
                sa_stats.append(b.stats())
            b.close()
        sa_ms = sum(x.ms_total for x in sa_stats) / len(sa_stats)
        line["with_suffix_array"] = {
            "value": round(bases / (sa_ms * 1e-3) / 1e6, 2), "unit": "Mbp/s", "ms_per_step": round(sa_ms, 3), "steps": sa_steps,
            "phase_ms": {"pack": round(sa_stats[-1].ms_pack, 2), "sort": round(sa_stats[-1].ms_sort, 2),
                         "refine": round(sa_stats[-1].ms_refine, 2), "wavelet": round(sa_stats[-1].ms_wt, 2)},
            "members_sorted": int(sa_stats[-1].refine_members),
            "note": "DSMFM_FLAG_KEEP_SA: every tie group sorted to the end; device time of dsmfm_build_device (events inside the library)"}

        # parity of what was timed: one more default-flags build through the host-buffer API, serialised and hashed, against
        # the digest of the .fmi the unmodified reference wrote for the same documents (tests/golden/fullsize.json)
        b = dsmfm.Builder(device=local, stream=stream.cuda_stream, expected_bytes=nbytes, flags=flags)
        b.append_batch(host_docs)
        sha, size = fmi_sha256(b.finish(), dsmfm)
        b.close()
        want = reference_digest(args.workload, kw)
        line["parity"] = {"sha256": sha, "fmi_bytes": size,
                          "matches": None if want is None else bool(want["fmi_sha256"] == sha and want["fmi_bytes"] == size),
                          "against": None if want is None else
                          "tests/golden/fullsize.json[%s]: %s" % (want["name"], want["reference"]),
                          "flags": flags}

    if world == 1 and not args.no_extras:
        line["fasta_e2e"] = fasta_front_end(args, kw, local, stream, torch, dsmfm, dsmgen)
        line["search"] = query_side(host_docs, local, stream, torch, dsmfm, args.steps)

    if world == 1 and not args.no_cpu_baseline:
        import tempfile
        try:
            with tempfile.TemporaryDirectory() as tmp:
                mbps, dt = cpu_reference_run(1, CPU_SAMPLE, tmp)
            line["cpu_baseline"] = {
                "value": round(mbps, 4), "unit": "Mbp/s", "cores": 1, "kind": "reference",
                "sample": "stock reference `builder` (single-threaded as shipped) on %d x %d-bp reads (%.0f Mbp, same generator "
                          "and error model as the workload), %.1f s" % (CPU_SAMPLE["n_reads"], CPU_SAMPLE["read_len"],
                                                                          CPU_SAMPLE["n_reads"] * CPU_SAMPLE["read_len"] / 1e6, dt)}
        except Exception:  # the compiled reference did not travel: time the oracle port instead
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle
            small = dict(CPU_SAMPLE, n_reads=20_000, genome_len=20_000)
            fa = dsmgen.fasta(**small).tobytes()
            t0 = time.perf_counter()
            oracle.build(fa)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {
                "value": round(small["n_reads"] * small["read_len"] / dt / 1e6, 4), "unit": "Mbp/s", "cores": 1,
                "kind": "port", "sample": "oracle/dsm_oracle.c on %d x %d-bp reads, %.1f s (oracle/_ref absent)"
                                          % (small["n_reads"], small["read_len"], dt)}
    real_stdout.write(json.dumps(line) + "\n")
    real_stdout.flush()
    if dist is not None:
        dist.destroy_process_group()
    if line.get("parity", {}).get("matches") is False:
        print("bench.py: the index that was timed differs from the reference's", file=sys.stderr)
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())
