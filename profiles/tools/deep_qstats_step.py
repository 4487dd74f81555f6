"""The deep-sample step with and without the strand / quality sums (DESIGN.md 5), on bench.py's deep shape: the 1 M-read
config-2 sample with every read --copies times (8 M reads), contiguous read ranges per rank.  One step is

    reset_async -> process_device (fused kernel [+ amp_qstats_kernel]) -> all-reduce(s) -> pack -> all-gather -> merge
    -> call_device [+ call_ivar_device]

timed with CUDA events on one stream; the plain step uses amp_allreduce_counts / amp_ins_pack_device / amp_ins_merge_packed,
the stats step amp_allreduce_qstats (three all-reduces) / amp_ins_pack_qstats_device / amp_ins_merge_packed_qstats.  The two
modes alternate, block by block.  The device error word is read after every step (outside the timed spans).  The fused kernel
and amp_qstats_kernel are timed apart in a torch.profiler pass of their own after the timed blocks.  Slots are sized as bench.py
sizes its own (32768 alleles, 2 MB of records per rank).  Rank 0 prints one JSON object with the GPU's name and power limit,
read in the same run, and writes it to --out when given.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29613 \\
        profiles/tools/deep_qstats_step.py [--steps K] [--copies C] [--out DIR]

Run from the repository root; N = 1 runs the same step with a one-rank communicator."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SPANS = ("process", "allreduce", "pack", "allgather", "merge", "call")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


class Leg:
    """One engine and its exchange over this rank's reads, with or without the sums."""

    def __init__(self, qstats, mine, tables, mpl, g, local, world, rank):
        from amplipy_b200 import dist as adist
        from amplipy_b200.engine import Engine
        from bench import L_GENOME
        self.qstats, self.world, self.rank = qstats, world, rank
        self.eng = Engine(ref_len=L_GENOME, primer_tables=tables, max_primer_len=mpl, device=local)
        if qstats:
            self.eng.enable_qstats()
        self.eng.set_reference(g)
        self.d = self.eng.upload(mine)
        self.eng.reserve(mine.n, int(mine.cig_off[-1]))
        self.ex = adist.DeepExchange(self.eng, cap_entries=1 << 15, cap_arena_bytes=2 << 20)

    def step(self, s, stream, evs=None):
        e, ex = self.eng, self.ex
        rec = (lambda i: evs[i].record(stream)) if evs else (lambda i: None)
        e.reset_async(s)
        rec(0)
        e.process_device(self.d, stream=s, qstats=self.qstats)
        rec(1)
        (e.allreduce_qstats if self.qstats else e.allreduce_counts)(ex.comm, s)
        rec(2)
        (e.ins_pack_qstats_device if self.qstats else e.ins_pack_device)(ex.send.data_ptr(), ex.cap_entries, ex.cap_arena, s)
        rec(3)
        ex.comm.allgather(ex.send.data_ptr(), ex.recv.data_ptr(), ex.slot_bytes, s)
        rec(4)
        (e.ins_merge_packed_qstats if self.qstats else e.ins_merge_packed)(ex.recv.data_ptr(), self.world, self.rank, ex.cap_entries,
                                                                          ex.cap_arena, s)
        rec(5)
        e.call_device(stream=s)
        if self.qstats:
            e.call_ivar_device(stream=s)
        rec(6)

    def close(self):
        self.ex.close()
        self.eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per mode and block")
    ap.add_argument("--blocks", type=int, default=3, help="alternating blocks per mode")
    ap.add_argument("--copies", type=int, default=8)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--out", help="directory for deep_qstats_step_n<N>.json (default: print only)")
    args = ap.parse_args()
    import torch.distributed as dist
    from amplipy_b200 import dist as adist
    from amplipy_b200 import synth
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len
    from bench import L_GENOME, make_workload
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    g, prim, base = make_workload(args.reads, 2, "illumina")
    tables = find_overlapping_primers(L_GENOME, prim, 0)
    mpl = max_primer_len(prim)
    first, count = adist.read_range(base.n, rank, world)
    sl = base.slice(first, first + count)
    mine = synth._reorder(sl, np.repeat(np.arange(sl.n, dtype=np.int64), args.copies))
    legs = {q: Leg(q, mine, tables, mpl, g, local, world, rank) for q in (False, True)}
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    spans = {q: [] for q in legs}
    errors = 0
    with torch.cuda.stream(stream):
        for q, leg in legs.items():
            for _ in range(3):
                leg.step(s, stream)
            torch.cuda.synchronize()
        for _ in range(args.blocks):
            for q, leg in legs.items():
                dist.barrier()
                for _ in range(args.steps):
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
                    leg.step(s, stream, ev)
                    errors |= leg.eng.error_flags()           # synchronises the device: after the step's last event
                    spans[q].append([ev[i].elapsed_time(ev[i + 1]) for i in range(6)])
        torch.cuda.synchronize()
        # kernel times from a profiler pass of its own
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for q, leg in legs.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    leg.step(s, stream)
                torch.cuda.synchronize()
            for ka in prof.key_averages():
                if "amp_trim_pileup" in ka.key or "amp_qstats_kernel" in ka.key:
                    key = ("qstats_pass_ms" if "amp_qstats_kernel" in ka.key else "fused_kernel_ms", q)
                    kern[key] = kern.get(key, 0.0) + ka.device_time_total / 1e3 / 5       # us over 5 steps -> ms per step
    # the slowest rank bounds every span
    res = {}
    for q in legs:
        a = np.array(spans[q]).mean(axis=0)
        tt = torch.tensor([a.sum()] + a.tolist() + [kern.get(("fused_kernel_ms", q), 0.0), kern.get(("qstats_pass_ms", q), 0.0)],
                          device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        v = tt.tolist()
        res["qstats" if q else "plain"] = dict(step_ms=v[0], **{k + "_ms": x for k, x in zip(SPANS, v[1:7])}, fused_kernel_ms=v[7],
                                               qstats_pass_ms=v[8], slot_bytes=legs[q].ex.slot_bytes,
                                               allreduce_bytes=int(6 * legs[q].eng.lpad * (16 if q else 4)))
    err = torch.tensor([errors], device="cuda", dtype=torch.int64)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    for leg in legs.values():
        leg.close()
    if rank == 0:
        out = {"gpu": gpu_info(), "ranks": world, "reads": base.n * args.copies, "steps": args.steps * args.blocks,
               "device_error_flags": int(err.item()), **res}
        print(json.dumps(out))
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "deep_qstats_step_n%d.json" % world), "w") as f:
                json.dump(out, f, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
