"""Where the time of bench.py's device-resident step goes: reset_async -> process_device -> call_device, the bench's own
workload, under torch.profiler (CUDA activities, in a run of its own).  Prints every device operation of one step with its
duration and the idle gap in front of it, their sums, and the host's enqueue time per step next to the GPU's step time
(the host stays ahead of the GPU while the first is the smaller).

    python profiles/tools/step_tail.py [--workload illumina|ont] [--reads N] [--steps K] [--out DIR]

Run from the repository root (or from a copy of another tree, to profile that tree's library)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="illumina", choices=["illumina", "ont"])
    ap.add_argument("--reads", type=int, default=0, help="0: the bench's default (1 M Illumina / 300 k ONT-like reads)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default="", help="directory for the per-step table (JSON)")
    args = ap.parse_args()
    import bench
    from amplipy_b200.engine import Engine
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len

    ont = args.workload == "ont"
    reads = args.reads or (300_000 if ont else 1_000_000)
    g, prim, b = bench.make_workload(reads, 2, args.workload)
    eng = Engine(ref_len=bench.L_GENOME, primer_tables=find_overlapping_primers(bench.L_GENOME, prim, 0),
                 max_primer_len=max_primer_len(prim), device=0, ins_slots=(1 << 24) if ont else 0,
                 ins_arena_bytes=(1 << 30) if ont else 0)
    eng.set_reference(g)
    d = eng.upload(b)
    eng.reserve(b.n, int(b.cig_off[-1]))
    stream = torch.cuda.Stream()
    s = stream.cuda_stream

    def step():
        eng.reset_async(s)
        eng.process_device(d, trim=True, pileup=True, stream=s)
        eng.call_device(stream=s)

    with torch.cuda.stream(stream):
        for _ in range(5):
            step()
        torch.cuda.synchronize()
        # host enqueue vs GPU step time, profiler off
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        enqueue_us = (time.perf_counter() - t0) / args.steps * 1e6
        ev1.record(stream)
        torch.cuda.synchronize()
        gpu_us = ev0.elapsed_time(ev1) / args.steps * 1e3

        eng.launches = 0
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                step()
            torch.cuda.synchronize()
        per_step_launches = eng.launches / args.steps

    dev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    dev.sort(key=lambda e: e.time_range.start)
    n_ops = len(dev) // args.steps
    assert n_ops * args.steps == len(dev), "device operations differ between steps: %d over %d steps" % (len(dev), args.steps)
    rows = []
    for k in range(n_ops):
        durs = [dev[j * n_ops + k].time_range.elapsed_us() for j in range(args.steps)]
        gaps = [dev[j * n_ops + k].time_range.start - dev[j * n_ops + k - 1].time_range.end for j in range(args.steps) if j * n_ops + k > 0]
        rows.append({"op": dev[k].name, "us": float(np.median(durs)), "gap_before_us": float(np.median(gaps)) if gaps else 0.0})
    span = (dev[-1].time_range.end - dev[0].time_range.start) / args.steps
    busy = sum(r["us"] for r in rows)
    name = torch.cuda.get_device_name(0)
    out = {"workload": args.workload, "reads": b.n, "device": name, "ops_per_step": n_ops, "launches_per_step": per_step_launches,
           "ops": rows, "busy_us": busy, "gaps_us": span - busy, "profiled_step_us": span, "gpu_step_us": gpu_us,
           "host_enqueue_us": enqueue_us}
    print("%s, %s, %d reads, %d device operations per step" % (name, args.workload, b.n, n_ops))
    for r in rows:
        print("  %8.1f us  (gap before %5.1f us)  %s" % (r["us"], r["gap_before_us"], r["op"][:110]))
    print("busy %.1f us + gaps %.1f us = %.1f us per profiled step; step %.1f us with the profiler off" % (busy, span - busy, span, gpu_us))
    print("host enqueue %.1f us per step (%s the GPU's %.1f us)" % (enqueue_us, "ahead of" if enqueue_us < gpu_us else "BEHIND", gpu_us))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "step_tail_%s.json" % args.workload), "w") as f:
            json.dump(out, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
