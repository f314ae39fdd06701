"""Run under torchrun (one rank per GPU): multigpu.build_sharded(..., samples=True) over documents spread across the
ranks; every rank writes its share of the `.fmi` and `.sa` files, rank 0 checks both against the oracle.  Used by
test_gpu_sharded_samples.py."""
import os
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "dsm-framework_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import cases
    import dsmfm
    import multigpu
    import oracle
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    box = [tempfile.mkdtemp(prefix="dsmfm_mgs_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    try:
        for it, (seed, rate, ranges) in enumerate([(1, 5, 1), (2, 124, 2), (3, 1, 1)]):
            docs, _ = oracle.fasta_to_docs(cases.rnd_fasta(seed, 800, 90, minlen=15, genome=2000))
            doc_list = docs.split(b"\0")[:-1]
            b, e = multigpu.block_of(len(doc_list), rank, world)
            mine = b"".join(d + b"\0" for d in doc_list[b:e])
            src = torch.frombuffer(bytearray(mine), dtype=torch.uint8).cuda() if mine else torch.empty(0, dtype=torch.uint8)
            engine = multigpu.CudaEngine(local, flags=dsmfm.FLAG_KEEP_SA, samplerate=rate)
            sb = multigpu.build_sharded(dist, src, engine, ranges_per_gpu=ranges, samples=True)
            prefix = os.path.join(box[0], "case%d" % it)
            sb.write(prefix)
            sb.write_samples(prefix)
            sb.close()
            dist.barrier()
            if rank == 0:
                with open(prefix + ".fmi", "rb") as f:
                    assert f.read() == oracle.fmi_from_docs(docs, rate), "seed %d: .fmi differs" % seed
                with open(prefix + ".sa", "rb") as f:
                    assert f.read() == oracle.sa_file_from_docs(docs, rate), "seed %d: .sa differs" % seed
        dist.barrier()
        if rank == 0:
            print("MULTIGPU_SAMPLES_OK world=%d" % world)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
