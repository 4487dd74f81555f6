"""Cost of the anchored deletion table (DESIGN.md 3.7, --ivar_deletions) on the TSV step: reset, process(..., qstats=True) through the
host path, call, call_ivar and, with the table, call_ivar_dels, timed with a host clock around the synchronous calls, without and
with the table, alternating.  Three workloads:
  * config 2: 1 M Illumina reads (bench.py's shape);
  * the ONT-like shape: 300 k reads;
  * the contention case: 1 M 150-base reads over one amplicon, every one carrying the same 9-base deletion at 11288-11296, so every
    event of the pass goes to one slot of the table.
Kernel times of amp_qstats_kernel / amp_qstats_dels_kernel / amp_ivar_dels_kernel come from torch.profiler in a pass of their own.
Prints one JSON object with the GPU's name and power limit, read in the same run.

    python profiles/tools/dels_step.py [--reps K] [--out DIR]

Run from the repository root."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from amplipy_b200 import synth  # noqa: E402
from amplipy_b200.batch import ReadBatch  # noqa: E402
from amplipy_b200.engine import Engine  # noqa: E402
from amplipy_b200.primers import find_overlapping_primers, max_primer_len  # noqa: E402

L = 29903


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def deletion_batch(g, n, at=11287, length=9, read_len=150, seed=3):
    """n reads of read_len bases starting in [at - 120, at - 20), each with `length` reference bases deleted from 0-based `at`."""
    rng = np.random.default_rng(seed)
    start = np.sort(rng.integers(at - 120, at - 20, n)).astype(np.int64)
    k = at - start                                              # bases before the deletion
    j = np.arange(read_len)[None, :]
    refpos = start[:, None] + j + np.where(j >= k[:, None], length, 0)
    code = np.frombuffer(b"\0" * 65 + bytes([1, 0, 2, 0, 0, 0, 4] + [0] * 12 + [8]), np.uint8)   # A C G T -> 1 2 4 8
    gb = np.frombuffer(g.encode(), np.uint8)
    nib = code[gb[refpos]]
    seq = ((nib[:, 0::2] << 4) | nib[:, 1::2]).astype(np.uint8).ravel()
    cig = np.stack([(k << 4) | 0, np.full(n, (length << 4) | 2), ((read_len - k) << 4) | 0], 1).astype(np.uint32).ravel()
    off = lambda w: (np.arange(n + 1, dtype=np.int64) * w).astype(np.uint32)
    flag = np.where(np.arange(n) % 2 == 1, 16, 0).astype(np.uint16)
    return ReadBatch(start.astype(np.int32), flag, np.zeros(n, np.int32), off(3), cig, off(read_len // 2), seq, off(read_len),
                     np.full(n * read_len, 35, np.uint8)).validate()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write DIR/dels_step.json")
    args = ap.parse_args()
    g = synth.random_genome(L, 7)
    primers, amps = synth.make_scheme(L, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    tables = find_overlapping_primers(L, prim, 0)
    work = {"cfg2": (synth.illumina_batch(g, amps, 1_000_000, seed=1), True),
            "ont": (synth.ont_batch(g, amps, 300_000, seed=4), True),
            "deep_deletion": (deletion_batch(g, 1_000_000), False)}
    out = {"gpu": gpu_info(), "reps": args.reps, "workloads": {}}
    for name, (b, trim) in work.items():
        big = name == "ont"
        engs = {}
        for dels in (False, True):
            e = Engine(ref_len=L, primer_tables=tables, max_primer_len=max_primer_len(prim), device=0,
                       ins_slots=(1 << 24) if big else 0, ins_arena_bytes=(1 << 30) if big else 0)
            e.enable_qstats()
            if dels:
                e.enable_dels(1 << 22)
            engs[dels] = e

        def step(e, dels):
            e.reset()
            e.process(b, trim=trim, pileup=True, qstats=True)
            e.call(g)
            e.call_ivar(1, 0.03)
            if dels:
                e.call_ivar_dels(1, 0.03)

        times = {False: [], True: []}
        for dels in (False, True):
            step(engs[dels], dels)                      # warm-up
        for _ in range(args.reps):
            for dels in (False, True):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                step(engs[dels], dels)
                torch.cuda.synchronize()
                times[dels].append((time.perf_counter() - t0) * 1e3)
        rec = {"reads": b.n}
        for dels in (False, True):
            t = sorted(times[dels])
            rec["step_ms_" + ("with" if dels else "without")] = {"median": round(t[len(t) // 2], 2), "min": round(t[0], 2), "max": round(t[-1], 2)}
        d = engs[True].dels()
        rec["alleles"] = int(len(d.count))
        rec["max_allele_count"] = int(d.count.max()) if len(d.count) else 0
        rec["error_flags"] = [engs[False].error_flags(), engs[True].error_flags()]
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for dels in (False, True):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    step(engs[dels], dels)
                torch.cuda.synchronize()
            for ev in prof.key_averages():
                m = re.search(r"(amp_\w+_kernel)", ev.key)
                if m and ("qstats" in m.group(1) or "dels" in m.group(1)):
                    kern[m.group(1)] = round(ev.device_time_total / 3 / 1000.0, 3)
        rec["kernel_ms_per_step"] = kern
        t0 = time.perf_counter()
        engs[True].call_ivar_dels(1, 0.03)
        rec["call_ivar_dels_ms"] = round((time.perf_counter() - t0) * 1e3, 2)
        out["workloads"][name] = rec
        for e in engs.values():
            e.close()
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dels_step.json"), "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
