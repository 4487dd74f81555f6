"""Cost of the iVar-format outputs (DESIGN.md 3.7) on bench.py's workloads, with CUDA events:
  * the device-resident step (reset_async -> process_device -> call_device) without and with AMP_MODE_QSTATS, alternating, on
    config 2 (1 M Illumina reads) and the ONT-like shape (300 k reads);
  * amp_qstats_kernel's own time, from torch.profiler in a run of its own;
  * amp_call_ivar_device on one sample and on a plate context of many samples.
Prints one JSON object with the GPU's name and power limit, read in the same run.

    python profiles/tools/ivar_step.py [--steps K] [--plate N] [--out DIR]

Run from the repository root."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def time_ms(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    out = []
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    out = sorted(a.elapsed_time(b) for a, b in ev)
    return {"median_ms": out[len(out) // 2], "min_ms": out[0], "max_ms": out[-1]}


def kernel_ms(fn, name, iters=10):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    tot = [e.device_time_total for e in prof.key_averages() if name in e.key]
    return (sum(tot) / iters / 1000.0) if tot else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--plate", type=int, default=96)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import bench
    from amplipy_b200.engine import Engine
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len

    out = {"gpu": gpu_info()}
    for kind, reads in (("illumina", 1_000_000), ("ont", 300_000)):
        ont = kind == "ont"
        g, prim, b = bench.make_workload(reads, 2, kind)
        eng = Engine(ref_len=bench.L_GENOME, primer_tables=find_overlapping_primers(bench.L_GENOME, prim, 0), max_primer_len=max_primer_len(prim),
                     device=0, ins_slots=(1 << 24) if ont else 0, ins_arena_bytes=(1 << 30) if ont else 0)
        eng.set_reference(g)
        eng.enable_qstats()
        d = eng.upload(b)
        s = torch.cuda.current_stream().cuda_stream

        def step(q):
            def f():
                eng.reset_async(s)
                eng.process_device(d, trim=True, pileup=True, stream=s, qstats=q)
                eng.call_device(stream=s)
            return f
        plain, stats = [], []
        for _ in range(3):                      # alternate the two forms
            plain.append(time_ms(step(False), args.steps))
            stats.append(time_ms(step(True), args.steps))
        r = {"reads": reads,
             "step_ms": [x["median_ms"] for x in plain], "step_qstats_ms": [x["median_ms"] for x in stats],
             "qstats_kernel_ms": kernel_ms(step(True), "amp_qstats_kernel"),
             "fused_kernel_ms": kernel_ms(step(False), "amp_trim_pileup")}
        eng.call_ivar_device(1, 0.03, 0.0, stream=s)
        r["ivar_call_ms"] = time_ms(lambda: eng.call_ivar_device(1, 0.03, 0.5, stream=s), args.steps)["median_ms"]
        r["ivar_kernel_ms"] = kernel_ms(lambda: eng.call_ivar_device(1, 0.03, 0.5, stream=s), "amp_ivar_kernel")
        r["call_kernel_ms"] = kernel_ms(lambda: eng.call_device(stream=s), "amp_call_kernel")
        torch.cuda.synchronize()
        assert eng.error_flags() == 0
        out[kind] = r
        eng.close()
        del d
        if not ont:
            # a plate: the same 100 k reads in every sample, one calling launch over all of them
            sub = b.take(np.arange(100_000))
            plate = Engine(ref_len=bench.L_GENOME, primer_tables=find_overlapping_primers(bench.L_GENOME, prim, 0),
                           max_primer_len=max_primer_len(prim), device=0, n_samples=args.plate, ins_slots=1 << 24)
            plate.set_reference(g)
            plate.enable_qstats()
            dd = plate.upload(sub)
            for k in range(args.plate):
                plate.process_device(dd, trim=True, pileup=True, sample=k, qstats=True)
            plate.call_device()
            plate.call_ivar_device(1, 0.03, 0.5)
            out["plate"] = {"samples": args.plate, "reads_per_sample": sub.n,
                            "call_ms": time_ms(lambda: plate.call_device(), 10)["median_ms"],
                            "ivar_call_ms": time_ms(lambda: plate.call_ivar_device(1, 0.03, 0.5), 10)["median_ms"]}
            assert plate.error_flags() == 0
            plate.close()
            del dd
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ivar_step.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
