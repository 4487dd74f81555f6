"""Multi-contig step on the GPU (DESIGN.md 3.8): plan kernel time and launches of a grouped 8-contig step next to config 2's
single-contig step at the same read count, the extra cost of an ungrouped (shuffled) batch, the per-contig launches with 256
small contigs, and `aio --multi_contig` file to file.  Kernel times come from torch.profiler over the timed steps; step times
from a host clock around work that ends in a device synchronise.

    python profiles/tools/contig_step.py [--reads 1000000] [--steps 10] [--out DIR]
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from amplipy_b200 import alnio, cli, synth  # noqa: E402
from amplipy_b200.batch import ReadBatch  # noqa: E402
from amplipy_b200.engine import Engine  # noqa: E402
from amplipy_b200.primers import find_overlapping_primers, max_primer_len  # noqa: E402

SEG_LENS = [2341, 2341, 2233, 1778, 1565, 1413, 1027, 890]


def contigs(lens, n_reads, seed=0):
    segs = []
    per = n_reads // len(lens)
    for k, L in enumerate(lens):
        g = synth.random_genome(L, 1000 + seed + k)
        primers, amps = synth.make_scheme(L, max(2, (L - 60) // 260), amp_len=300, seed=2000 + seed + k)
        segs.append(dict(id="seg%d" % (k + 1), g=g, L=L, primers=primers, prim=sorted((s, e) for s, e, _ in primers),
                         b=synth.illumina_batch(g, amps, per, seed=3000 + seed + k)))
    b = ReadBatch.concat([s["b"] for s in segs])
    sid = np.concatenate([np.full(s["b"].n, k, np.int32) for k, s in enumerate(segs)])
    return segs, b, sid


def multi_engine(segs):
    e = Engine(ref_len=max(s["L"] for s in segs), n_samples=len(segs))
    for k, s in enumerate(segs):
        e.set_scheme(k, s["prim"], 0, ref_len=s["L"])
        e.set_sample_reference(k, s["g"])
    return e


def kernel_table(fn, steps):
    """{kernel name: (launches per step, us per step)} over `steps` calls of fn, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    acc = collections.defaultdict(lambda: [0, 0.0])
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower():
            nm = ev.name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0].split("<")[0]
            acc[nm][0] += 1
            acc[nm][1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    return {k: (v[0] / steps, round(v[1] / steps, 1)) for k, v in sorted(acc.items())}


def wall(fn, steps):
    import torch
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return round((time.perf_counter() - t) / steps * 1e6, 1)


def device_step(eng, d, sid_t, trim=True):
    """plan + process of a batch already in HBM (what Engine.process_contigs runs after its upload)."""
    import ctypes
    from amplipy_b200 import engine as em
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    db = em.AmpBatch(0, d["n"], p(d["pos"]), p(d["flag"]), p(d["tlen"]), p(d["cig_off"]), p(d["cigar"]), p(d["seq_off"]), p(d["seq"]),
                     p(d["qual_off"]), p(d["qual"]))
    to = em.AmpTrimOut(p(d["o_pos"]), p(d["o_ncig"]), p(d["o_flags"]), p(d["o_cigar"]))
    launches = 0

    def step():
        nonlocal launches
        plan = em.ContigPlan(eng.n_samples)
        em._check(eng.lib.amp_contig_plan_device(eng._ctx, ctypes.byref(db), p(sid_t), ctypes.byref(plan.c)), "plan")
        launches = int(eng.lib.amp_last_launches(eng._ctx))
        em._check(eng.lib.amp_process_contigs(eng._ctx, em.MODE_TRIM | em.MODE_PILEUP, ctypes.byref(to) if trim else None, None), "process")
        launches += int(eng.lib.amp_last_launches(eng._ctx))
        step.grouped = plan.grouped
    step()
    return step, lambda: launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    dev = torch.device("cuda", 0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"gpu": q.stdout.strip() or torch.cuda.get_device_name(0), "reads": a.reads}

    # config 2's single-contig step at the same read count (fused kernel on a batch in HBM)
    G = 29903
    g = synth.random_genome(G, 7)
    primers, amps = synth.make_scheme(G, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    b2 = synth.illumina_batch(g, amps, a.reads, seed=1)
    e2 = Engine(ref_len=G, primer_tables=find_overlapping_primers(G, prim, 0), max_primer_len=max_primer_len(prim))
    d2 = e2.upload(b2)
    one = lambda: e2.process_device(d2, trim=True, pileup=True)
    out["single_contig"] = {"kernels": kernel_table(one, a.steps), "step_us": wall(one, a.steps)}
    e2.close()

    for name, lens in (("8_contigs", SEG_LENS), ("256_contigs", [int(x) for x in np.random.default_rng(5).integers(400, 2500, 256)])):
        segs, b, sid = contigs(lens, a.reads)
        for order_name, order in (("grouped", np.arange(b.n)), ("shuffled", np.random.default_rng(9).permutation(b.n))):
            if name == "256_contigs" and order_name == "shuffled":
                continue
            eng = multi_engine(segs)
            bb = b.take(order)
            d = eng.upload(bb)
            sid_t = torch.from_numpy(np.ascontiguousarray(sid[order])).to(dev)
            step, nl = device_step(eng, d, sid_t)
            assert step.grouped == (order_name == "grouped")
            out["%s_%s" % (name, order_name)] = {"kernels": kernel_table(step, a.steps), "step_us": wall(step, a.steps), "launches": nl()}
            eng.close()

    # file to file: aio --multi_contig on the 8-contig BAM
    segs, b, sid = contigs(SEG_LENS, a.reads)
    with tempfile.TemporaryDirectory() as td:
        j = lambda n: os.path.join(td, n)
        hdr = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (s["id"], s["L"]) for s in segs) + "@PG\tID:synth\tPN:synth\tVN:1\n"
        alnio.write_bam(j("in.bam"), hdr, [(s["id"], s["L"]) for s in segs], b, refid=sid)
        with open(j("ref.fas"), "w") as f:
            f.write("".join(">%s\n%s\n" % (s["id"], s["g"]) for s in segs))
        with open(j("p.bed"), "w") as f:
            f.write("".join("%s\t%d\t%d\t%s\n" % (s["id"], st, en, nm) for s in segs for st, en, nm in s["primers"]))
        times = []
        for r in range(3):
            t = time.perf_counter()
            cli.main(["aio", "--multi_contig", "-i", j("in.bam"), "-p", j("p.bed"), "-r", j("ref.fas"), "-ot", j("o%d.bam" % r),
                      "-ov", j("o%d.vcf" % r), "-oc", j("o%d.fas" % r)])
            times.append(round(time.perf_counter() - t, 3))
        out["aio_8_contigs_file_s"] = times
        out["bam_mb"] = round(os.path.getsize(j("in.bam")) / 1e6, 1)
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "contig_step.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
