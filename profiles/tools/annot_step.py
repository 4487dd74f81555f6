"""Codon annotation on the GPU (DESIGN.md 3.9): set_features + annotate (table build, translations and the host copy) for one
29,903-base sample and for a 384-sample plate with per-sample references, the kernels' own times, and `aio --output_tsv` on a
config-2 BAM with and without `--gff`.  Kernel times come from torch.profiler; call times from a host clock around calls that end
in a device synchronise (amp_annotate and amp_annot_host both synchronise).

    python profiles/tools/annot_step.py [--reps 10] [--reads 1000000] [--out DIR]
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
from amplipy_b200.engine import Engine  # noqa: E402
from amplipy_b200.gff import Feature  # noqa: E402

G = 29903
# a SARS-CoV-2-like CDS layout (NCBI's MN908947.3 coordinates, 0-based half-open): ORF1ab with its -1 frameshift, nested ORFs
CDS = [("ORF1ab", [(265, 13468), (13467, 21555)]), ("ORF1a", [(265, 13483)]), ("S", [(21562, 25384)]), ("ORF3a", [(25392, 26220)]),
       ("E", [(26244, 26472)]), ("M", [(26522, 27191)]), ("ORF6", [(27201, 27387)]), ("ORF7a", [(27393, 27759)]),
       ("ORF7b", [(27755, 27887)]), ("ORF8", [(27893, 28259)]), ("N", [(28273, 29533)]), ("ORF9b", [(28283, 28577)]),
       ("ORF10", [(29557, 29674)])]
FEATURES = [Feature(n, "ref", 1, 0, sg) for n, sg in CDS]


def kernel_table(fn, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    acc = collections.defaultdict(lambda: [0, 0.0])
    for ev in prof.events():
        if ev.device_type.name == "CUDA":
            nm = ev.name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0].split("<")[0]
            acc[nm][0] += 1
            acc[nm][1] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    return {k: (v[0] / reps, round(v[1] / reps, 1)) for k, v in sorted(acc.items())}


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return {"median_ms": round(float(np.median(ts)), 3), "min_ms": round(min(ts), 3), "max_ms": round(max(ts), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"gpu": q.stdout.strip()}
    g = synth.random_genome(G, 7)

    # one sample
    e = Engine(ref_len=G)
    e.set_reference(g)

    def one():
        e.set_features(0, FEATURES)
        return e.annotate()
    out["one_sample"] = {"set_features_annotate": timed(one, a.reps), "entries": int(len(one().feat)), "kernels_us": kernel_table(one, a.reps)}
    e.close()

    # a 384-sample plate, a reference of its own per sample
    S = 384
    rng = np.random.default_rng(1)
    p = Engine(ref_len=G, n_samples=S)
    base = np.frombuffer(g.encode(), np.uint8)
    for s in range(S):
        r = base.copy()
        m = rng.random(G) < 0.001
        r[m] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(m.sum()))]
        p.set_sample_reference(s, r.tobytes())

    def plate():
        for s in range(S):
            p.set_features(s, FEATURES)
        return p.annotate()
    out["plate_384"] = {"set_features_annotate": timed(plate, a.reps), "entries": int(len(plate().feat)),
                        "kernels_us": kernel_table(plate, a.reps)}
    p.close()
    print(json.dumps(out, indent=1), flush=True)

    # file to file: aio --output_tsv on a config-2 BAM, with and without --gff, alternating
    primers, amps = synth.make_scheme(G, 98, seed=2)
    snvs = [(1000 + 2800 * i, "ACGT"[i % 4], af) for i, af in enumerate([1.0, 0.9, 0.75, 0.5, 0.4, 0.3, 0.2, 0.1, 0.05, 0.05])]
    b = synth.illumina_batch(g, amps, a.reads, seed=1, snvs=snvs)
    with tempfile.TemporaryDirectory() as td:
        j = lambda n: os.path.join(td, n)
        alnio.write_bam(j("in.bam"), "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:%d\n@PG\tID:synth\tPN:synth\tVN:1\n" % G, [("ref", G)], b)
        synth.write_fasta(j("ref.fas"), "ref", g)
        synth.write_bed(j("p.bed"), primers, rname="ref")
        with open(j("a.gff"), "w") as f:
            f.write("##gff-version 3\n" + "".join("ref\tx\tCDS\t%d\t%d\t.\t+\t0\tID=%s\n" % (lo + 1, hi, n) for n, sg in CDS for lo, hi in sg))
        times = {"plain": [], "gff": []}
        for r in range(4):
            for tag in ("plain", "gff"):
                extra = ["--gff", j("a.gff")] if tag == "gff" else []
                t = time.perf_counter()
                cli.main(["aio", "-i", j("in.bam"), "-p", j("p.bed"), "-r", j("ref.fas"), "-ot", j("o%s%d.bam" % (tag, r)), "-ov",
                          j("o%s%d.vcf" % (tag, r)), "-oc", j("o%s%d.fas" % (tag, r)), "--output_tsv", j("o%s%d.tsv" % (tag, r))] + extra)
                times[tag].append(round(time.perf_counter() - t, 3))
        out["aio_output_tsv_s"] = times
        out["tsv_rows"] = {tag: sum(1 for _ in open(j("o%s0.tsv" % tag))) - 1 for tag in ("plain", "gff")}
        out["bam_mb"] = round(os.path.getsize(j("in.bam")) / 1e6, 1)
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "annot_step.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
