"""Run under torchrun (NCCL): a read-sharded deep sample with the anchored deletion table must give, on every rank, the deletion
alleles (count, rev, qsum, mq, PVAL by their bytes) and TSV rows of one GPU over all the reads (computed on rank 0), and all ranks
must agree.  The exchange (DeepExchange.run: the all-reduce, the insertion slots and the deletion slots through NCCL) runs at
every world size, one included.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29613 tests/dist_gpu_dels_check.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def outputs(eng, g):
    from amplipy_b200 import ivar
    res = eng.call(g)
    d = eng.call_ivar_dels(1, 0.03)
    alleles = [(int(d.sample[k]), int(d.anchor[k]), int(d.len[k]), int(d.count[k]), int(d.rev[k]), int(d.qsum[k]), int(d.mq[k]),
                np.float64(d.pval[k]).tobytes()) for k in range(len(d.count))]
    rows = [ivar.format_row(r) for r in ivar.tsv_rows(res, eng.insertions(), eng.call_ivar(1, 0.03, 0.0), eng.qstats(), "ref", g,
                                                      eng.counts(), dels=d)]
    return alleles, rows


def main():
    import torch
    import torch.distributed as dist
    from amplipy_b200 import synth
    from amplipy_b200 import dist as adist
    from amplipy_b200.engine import Engine
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = 29903
    g = synth.random_genome(L, 7)
    primers, amps = synth.make_scheme(L, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    tables = find_overlapping_primers(L, prim, 0)
    mpl = max_primer_len(prim)
    for kind, b, big in (("cfg2", synth.illumina_batch(g, amps, 400_000, seed=77), False),
                         ("ont", synth.ont_batch(g, amps, 20_000, seed=4), True)):
        kw = dict(ref_len=L, primer_tables=tables, max_primer_len=mpl, ins_slots=(1 << 24) if big else 0,
                  ins_arena_bytes=(1 << 30) if big else 0)
        eng = Engine(device=local, **kw)
        eng.enable_qstats()
        eng.enable_dels(1 << 20)
        ex = adist.DeepExchange(eng, cap_entries=1 << 18, cap_arena_bytes=64 << 20, cap_dels=1 << 18)
        first, count = adist.read_range(b.n, rank, world)
        eng.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)
        ex.run(None)
        torch.cuda.synchronize(local)
        ex.close()
        assert eng.error_flags() == 0, "%s: device error 0x%x on rank %d" % (kind, eng.error_flags(), rank)
        got = outputs(eng, g)
        if rank == 0:
            solo = Engine(device=local, **kw)
            solo.enable_qstats()
            solo.enable_dels(1 << 20)
            solo.process(b, trim=True, pileup=True, qstats=True)
            want = outputs(solo, g)
            assert got[0] == want[0] and len(want[0]) > 0, "%s: deletion alleles differ from one GPU" % kind
            assert got[1] == want[1], "%s: TSV rows differ from one GPU" % kind
            solo.close()
        h = hashlib.sha256(repr(got).encode()).digest()[:8]
        chk = torch.tensor([int.from_bytes(h, "little") >> 1, len(got[0]), len(got[1])], device="cuda", dtype=torch.int64)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), "%s: ranks disagree after the exchange" % kind
        if rank == 0:
            print("dist_gpu_dels_check ok: world=%d %s, %d deletion alleles, %d TSV rows" % (world, kind, len(got[0]), len(got[1])))
        eng.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
