"""Multi-GPU sharding of the path (one process per GPU, torch.distributed for the plumbing).

Two natural partitions (SURVEY.md section 8e):

* plate  -- samples are independent: sample i goes to rank i % world; no data-path collective at all.
* deep   -- one sample, contiguous read ranges per rank.  Trim outputs are per read (no exchange); each
            rank accumulates a private count matrix and insertion table; then ONE all-reduce (sum, int32)
            of the [6, lpad] matrix over NVLink/NVSwitch and ONE all-gather of the ranks' insertion tables, packed on
            the device into fixed-size slots, merged into every rank's table by one kernel.  Nothing passes through
            the host.  Integer sums => the result is independent of the partition and bit-identical to one GPU.

On CUDA engines the exchange runs through the C ABI (amp_allreduce_counts, amp_ins_pack_device, amp_nccl_allgather,
amp_ins_merge_packed) on a communicator made by ``DeepExchange``; engines without that entry point (the CPU emulation
used by the gloo tests) take the torch.distributed form of the same two steps.  An engine with the strand / quality sums
(``enable_qstats``) exchanges them too: the all-reduce also sums its rev / qsum matrices and every exchanged insertion
allele carries its ins_rev / ins_qsum / ins_head (the *_qstats entry points), so the iVar outputs of every rank are those
of one GPU over all the reads.  An engine with the anchored deletion table (``enable_dels``) also packs, gathers and merges
that table (amp_dels_pack_device, amp_nccl_allgather, amp_dels_merge_packed; its sums are integers too).

The reference has no counterpart (single sequential loop, AmpliPy.py:896)."""
import numpy as np


def plate_assignment(n_samples, rank, world):
    """Samples owned by `rank` (round-robin)."""
    return list(range(rank, n_samples, world))


def read_range(n_reads, rank, world):
    """Contiguous [first, first + count) slice of a coordinate-sorted batch for `rank`."""
    first = (n_reads * rank) // world
    last = (n_reads * (rank + 1)) // world
    return first, last - first


class DeepExchange:
    """Device-side exchange step of the deep-sample mode for one CUDA engine: an NCCL communicator of its own (created
    through the C ABI; the id travels over the torch.distributed group once) and the two slot buffers, allocated once.

    cap_entries / cap_arena_bytes: capacity of a rank's slot (distinct insertion alleles / bytes of their records); a
    table that does not fit raises the engine's TABLE_FULL / ARENA_FULL error flag.  The engine's strand / quality sums,
    when it has them at construction (``engine.qstats_enabled``), travel with the counts and the alleles.  So does its anchored
    deletion table (``engine.dels_enabled``), in slots of cap_dels alleles; a table that does not fit raises DELS_FULL."""

    def __init__(self, engine, group=None, cap_entries=1 << 16, cap_arena_bytes=4 << 20, cap_dels=1 << 16):
        import torch
        import torch.distributed as dist
        from .engine import NcclComm
        self.engine = engine
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.cap_entries, self.cap_arena = int(cap_entries), int(cap_arena_bytes)
        self.qstats = engine.qstats_enabled
        slot_bytes = engine.ins_slot_bytes_qstats if self.qstats else engine.ins_slot_bytes
        self.slot_bytes = slot_bytes(self.cap_entries, self.cap_arena)
        dev = torch.device("cuda", engine.device)
        self.send = torch.zeros(self.slot_bytes, dtype=torch.uint8, device=dev)
        self.recv = torch.zeros(self.slot_bytes * self.world, dtype=torch.uint8, device=dev)
        self.dels = getattr(engine, "dels_enabled", False)
        if self.dels:
            self.cap_dels = int(cap_dels)
            self.dels_bytes = engine.dels_slot_bytes(self.cap_dels)
            self.dels_send = torch.zeros(self.dels_bytes, dtype=torch.uint8, device=dev)
            self.dels_recv = torch.zeros(self.dels_bytes * self.world, dtype=torch.uint8, device=dev)
        self.comm = NcclComm.from_torch_group(engine.device, group)

    def run(self, stream=None):
        """all-reduce of the counts + exchange of the insertion tables, asynchronous on ``stream`` (a raw cudaStream_t)."""
        e = self.engine
        if self.qstats:
            allreduce, pack, merge = e.allreduce_qstats, e.ins_pack_qstats_device, e.ins_merge_packed_qstats
        else:
            allreduce, pack, merge = e.allreduce_counts, e.ins_pack_device, e.ins_merge_packed
        allreduce(self.comm, stream)
        pack(self.send.data_ptr(), self.cap_entries, self.cap_arena, stream)
        self.comm.allgather(self.send.data_ptr(), self.recv.data_ptr(), self.slot_bytes, stream)
        merge(self.recv.data_ptr(), self.world, self.rank, self.cap_entries, self.cap_arena, stream)
        if self.dels:
            e.dels_pack_device(self.dels_send.data_ptr(), self.cap_dels, stream)
            self.comm.allgather(self.dels_send.data_ptr(), self.dels_recv.data_ptr(), self.dels_bytes, stream)
            e.dels_merge_packed(self.dels_recv.data_ptr(), self.world, self.rank, self.cap_dels, stream)

    def close(self):
        self.comm.close()


def allreduce_counts(engine, group=None):
    """torch.distributed form: sum the per-rank count matrices in place (every rank ends up with the total), and the rev /
    qsum matrices of an engine with the strand / quality sums."""
    import torch.distributed as dist
    t = engine.counts_tensor()
    if t.is_cuda:
        import torch
        torch.cuda.synchronize(t.device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    if getattr(engine, "qstats_enabled", False):
        for s in engine.qstats_tensors():
            dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
    return t


def allgather_insertions(engine, group=None):
    """torch.distributed form (host arrays): exchange the distinct insertion alleles of every rank and merge the others'
    into the local table.  Used by engines without the packed device-side exchange (the CPU emulation)."""
    import torch.distributed as dist
    rank = dist.get_rank(group)
    world = dist.get_world_size(group)
    ins = engine.insertions()
    mine = (np.asarray(ins.sample), np.asarray(ins.pos), np.asarray(ins.count), np.asarray(ins.str_off), np.asarray(ins.chars))
    if getattr(engine, "qstats_enabled", False):     # each allele's strand / quality sums travel with it
        qs = engine.qstats()
        mine += (np.asarray(qs.ins_rev), np.asarray(qs.ins_qsum), np.asarray(qs.ins_head))
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=group)
    for r, part in enumerate(gathered):
        if r != rank and len(part[1]):
            engine.merge_insertions(*part)
    return engine.insertions()


def allgather_dels(engine, group=None):
    """torch.distributed form (host arrays) of the deletion-table exchange: every rank's anchored deletion alleles gathered, the
    others' merged into the local table (engines with ``dels_enabled``)."""
    import torch.distributed as dist
    rank = dist.get_rank(group)
    gathered = [None] * dist.get_world_size(group)
    dist.all_gather_object(gathered, engine.dels(), group=group)
    for r, part in enumerate(gathered):
        if r != rank and len(part.count):
            engine.merge_dels(part)
    return engine.dels()


def process_deep_sample(engine, batch, trim=True, pileup=True, sample=0, group=None, exchange=None, qstats=False):
    """Read-sharded processing of one sample: local kernel on this rank's read range, then the exchange step.
    Returns this rank's TrimResult (valid for its own range of reads only; the other reads' flags are 0).
    ``exchange``: a DeepExchange to reuse (CUDA engines); one is created and closed when it is None.
    ``qstats``: the strand / quality pass runs on the same reads (engine.enable_qstats first); the exchange carries the sums
    whenever the engine has them.  Without it, engine.process is called as before, so engines without the pass work unchanged."""
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    first, count = read_range(batch.n, rank, world)
    t = engine.process(batch, trim=trim, pileup=pileup, sample=sample, first=first, n=count, **({"qstats": True} if qstats else {}))
    if pileup and world > 1:
        if hasattr(engine, "ins_pack_device"):
            import torch
            ex = exchange or DeepExchange(engine, group)
            ex.run(None)
            torch.cuda.synchronize(engine.device)
            if exchange is None:
                ex.close()
        else:
            allreduce_counts(engine, group)
            allgather_insertions(engine, group)
            if getattr(engine, "dels_enabled", False):
                allgather_dels(engine, group)
    return t, (first, count)
