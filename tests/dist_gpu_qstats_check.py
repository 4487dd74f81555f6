"""Run under torchrun on >= 2 GPUs (NCCL): a read-sharded deep sample with the strand / quality sums must give, on every
rank, the calling outputs, iVar outputs (p-values compared by their bytes, IUPAC codes) and TSV rows of one GPU over all the
reads (computed on rank 0), and all ranks must agree.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29612 tests/dist_gpu_qstats_check.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CALL_FIELDS = ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask")


def outputs(eng, g):
    """Per-position arrays as bytes and per-allele outputs keyed by (sample, pos, string): the export order depends on the order
    in which the table was filled."""
    from amplipy_b200 import ivar
    res = eng.call(g)
    ins, qs = eng.insertions(), eng.qstats()
    iv = eng.call_ivar(1, 0.03, 0.0)
    ivc = eng.call_ivar(10, 0.0, 0.75)
    # top_id >= 6 names an insertion allele by its export index: compare its string instead
    top = [t if t < 6 else ins.strs[t - 6] for t in res.top_id.tolist()]
    per_pos = [np.ascontiguousarray(getattr(res, f)).tobytes() for f in CALL_FIELDS] + \
        [top, iv.fixed_mq.tobytes(), iv.fixed_pval.tobytes(), iv.iupac.tobytes(), ivc.iupac.tobytes(), eng.counts().tobytes(),
         qs.rev.tobytes(), qs.qsum.tobytes()]
    per_allele = sorted(((int(ins.sample[k]), int(ins.pos[k]), ins.strs[k]),
                         (int(ins.count[k]), float(res.ins_freq[k]).hex(), int(res.ins_rank[k]), int(res.ins_alt[k]), int(qs.ins_rev[k]),
                          int(qs.ins_qsum[k]), int(qs.ins_head[k]), int(iv.ins_mq[k]), np.float64(iv.ins_pval[k]).tobytes()))
                        for k in range(ins.k))
    # the TSV as the command line writes it (PVAL by repr: exact)
    rows = [ivar.format_row(r) for r in ivar.tsv_rows(res, ins, iv, qs, "ref", g, eng.counts())]
    return per_pos, per_allele, rows


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
    for kind, b, big in (("cfg2", synth.illumina_batch(g, amps, 400_000, seed=77, p_ins=0.05), False),
                         ("ont", synth.ont_batch(g, amps, 20_000, seed=4), True)):
        kw = dict(ref_len=L, primer_tables=tables, max_primer_len=mpl, ins_slots=(1 << 24) if big else 0,
                  ins_arena_bytes=(1 << 30) if big else 0)
        eng = Engine(device=local, **kw)
        eng.enable_qstats()
        ex = adist.DeepExchange(eng, cap_entries=1 << 18, cap_arena_bytes=64 << 20)
        adist.process_deep_sample(eng, b, qstats=True, exchange=ex)
        ex.close()
        assert eng.error_flags() == 0, "%s: device error 0x%x on rank %d" % (kind, eng.error_flags(), rank)
        got = outputs(eng, g)
        if rank == 0:
            solo = Engine(device=local, **kw)
            solo.enable_qstats()
            solo.process(b, trim=True, pileup=True, qstats=True)
            want = outputs(solo, g)
            assert got[0] == want[0], "%s: per-position outputs differ from one GPU" % kind
            assert got[1] == want[1], "%s: per-allele outputs differ from one GPU" % kind
            assert got[2] == want[2] and len(want[2]) > 0, "%s: TSV rows differ from one GPU" % kind
            solo.close()
        h = hashlib.sha256(repr(got).encode()).digest()[:8]
        chk = torch.tensor([int.from_bytes(h, "little") >> 1, len(got[1]), len(got[2])], device="cuda", dtype=torch.int64)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), "%s: ranks disagree after the exchange" % kind
        if rank == 0:
            print("dist_gpu_qstats_check ok: world=%d %s, %d alleles, %d TSV rows" % (world, kind, len(got[1]), len(got[2])))
        eng.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
