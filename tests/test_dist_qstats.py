"""The deep-sample exchange of the strand / quality sums (DESIGN.md 3.7, 5): after the exchange every rank of a read-sharded
sample holds the counts, insertion alleles, rev / qsum and per-allele ins_rev / ins_qsum / ins_head of one context over all the
reads, so its iVar outputs are the single-GPU ones.

CPU: the pack and merge bodies of amp_exchange.cuh on the emulator over 2-4 "ranks", and the torch.distributed (gloo) form of
dist.process_deep_sample at world size 2 and 3.  GPU: the *_qstats entry points across contexts on one device, a one-rank NCCL
communicator, the state errors, and the plain exchange left as it was.  Per-allele outputs are compared keyed by
(sample, pos, string): the export order depends on the order in which each table was filled."""
import ctypes
import os
import shutil
import socket
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import emu_dist_driver
import emu_driver
import golden_io
import parity
from amplipy_b200 import calling, ivar, synth
from amplipy_b200.primers import find_overlapping_primers, max_primer_len

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HERE = os.path.join(ROOT, "tests")
TABLE_FULL, ARENA_FULL = 16, 32
FUZZ_L = 29903


# ---------------------------------------------------------------------------------------------------------------- fixtures
def load_fixture(name):
    """(batch, engine kwargs, reference, calling params) of a golden case or of the seeded indel-rich fuzz sample."""
    if name == "fuzz":
        g = synth.random_genome(FUZZ_L, 3)
        primers, amps = synth.make_scheme(FUZZ_L, 98, seed=4)
        prim = [(s, e) for s, e, _ in primers]
        b = synth.illumina_batch(g, amps, 3000, seed=31, p_ins=0.08, p_del=0.08)
        kw = dict(ref_len=FUZZ_L, primer_tables=find_overlapping_primers(FUZZ_L, prim, 0), max_primer_len=max_primer_len(prim))
        p = {"min_depth_consensus": 10, "min_freq_consensus": 0.0, "min_depth_variants": 1, "min_freq_variants": 0.03,
             "unknown_symbol": "N"}
        return b, kw, g, p
    b, meta, arr = golden_io.load_case(name)
    return b, parity.engine_kwargs(meta), bytes(arr["ref_seq"]).decode(), meta["params"]


FIXTURES = ["cfg3_deep_alt", "cfg4_ont", "fuzz"]


@pytest.fixture(autouse=True)
def _emulator(monkeypatch):
    emu_dist_driver.install(monkeypatch)


def emu_engine(kw, qstats=True):
    """An emulated context with the sums enabled; ``qstats=False``: the plain EmuEngine, which has no stats surface at all."""
    if not qstats:
        return emu_driver.EmuEngine(**kw, ins_slots=1 << 18, ins_arena_bytes=1 << 24)
    e = emu_dist_driver.EmuQstatsEngine(**kw, ins_slots=1 << 18, ins_arena_bytes=1 << 24)
    e.enable_qstats()
    return e


def keyed(eng, sample=0):
    """{(sample, pos, string): (count, ins_rev, ins_qsum, ins_head)} of every allele in the table."""
    ins, qs = eng.insertions(), eng.qstats(sample)
    return {(int(ins.sample[k]), int(ins.pos[k]), ins.strs[k]): (int(ins.count[k]), int(qs.ins_rev[k]), int(qs.ins_qsum[k]), int(qs.ins_head[k]))
            for k in range(ins.k)}


def read_ranges(n, k):
    return [(n * r // k, n * (r + 1) // k - n * r // k) for r in range(k)]


def ivar_outputs(eng, ref, p, ref_id="ref"):
    """What the command line writes from a stats context: the TSV lines and the IUPAC consensus at thresholds 0 and 0.75."""
    res = eng.call(ref, p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"], p["min_freq_variants"])
    ins, qs, counts = eng.insertions(), eng.qstats(), eng.counts()
    iv = eng.call_ivar(p["min_depth_variants"], p["min_freq_variants"], 0.0)
    rows = [ivar.format_row(r) for r in ivar.tsv_rows(res, ins, iv, qs, ref_id, ref, counts)]
    cons = []
    for t in (0.0, 0.75):
        ivc = eng.call_ivar(p["min_depth_consensus"], p["min_freq_consensus"], t)
        cons.append(calling.consensus_string(res, ins, 0, p["unknown_symbol"], iupac=ivc.iupac))
    return rows, cons


# ---------------------------------------------------------------------------------------------------------------- CPU: emulated pack / merge
def _sharded(b, kw, k):
    engs = []
    for first, count in read_ranges(b.n, k):
        e = emu_engine(kw)
        e.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)
        engs.append(e)
    return engs


def _caps(engs):
    return (max(int(emu_dist_driver.lib().emu_ins_count(e._h)) for e in engs),
            max(int(emu_dist_driver.lib().emu_ins_chars(e._h)) for e in engs))


def _pack_all(engs, cap_e, cap_a):
    words = engs[0].ins_slot_bytes_qstats(cap_e, cap_a) // 8
    slots = np.zeros(len(engs) * words, np.uint64)
    for r, e in enumerate(engs):
        e.ins_pack_qstats(slots[r * words:(r + 1) * words], cap_e, cap_a)
    return slots, words


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("name", FIXTURES)
def test_emulated_pack_merge_equals_one_context(name, k):
    b, kw, ref, p = load_fixture(name)
    solo = emu_engine(kw)
    solo.process(b, trim=True, pileup=True, qstats=True)
    want, want_q = keyed(solo), solo.qstats()
    engs = _sharded(b, kw, k)
    # the matrices, summed as the all-reduce sums them
    counts = sum(e.counts_tensor().numpy().astype(np.int64) for e in engs)
    rev = sum(e.qstats_tensors()[0].numpy().astype(np.int64) for e in engs)
    qsum = sum(e.qstats_tensors()[1].numpy() for e in engs)
    L = kw["ref_len"]
    assert np.array_equal(counts[0, :, :L], solo.counts())
    assert np.array_equal(rev[0, :, :L], want_q.rev) and np.array_equal(qsum[0, :, :L], want_q.qsum)
    cap_e, cap_a = _caps(engs)                      # every slot sized for the largest table: that one fits exactly
    assert cap_e > 0
    slots, _ = _pack_all(engs, cap_e, cap_a)
    for r, e in enumerate(engs):
        e.ins_merge_packed_qstats(slots, k, r, cap_e, cap_a)
        assert e.error_flags() == 0
        assert keyed(e) == want, (name, k, r)


@pytest.mark.parametrize("short", ["entry", "arena"])
@pytest.mark.parametrize("name", ["cfg4_ont", "fuzz"])
def test_emulated_pack_overflow_packs_empty(name, short):
    b, kw, ref, p = load_fixture(name)
    engs = _sharded(b, kw, 2)
    n0, a0 = int(emu_dist_driver.lib().emu_ins_count(engs[0]._h)), int(emu_dist_driver.lib().emu_ins_chars(engs[0]._h))
    cap_e, cap_a = (n0 - 1, a0) if short == "entry" else (n0, a0 - 8)
    before = keyed(engs[1])
    words = engs[0].ins_slot_bytes_qstats(cap_e, cap_a) // 8
    slots = np.full(2 * words, 0xA5A5A5A5A5A5A5A5, np.uint64)
    engs[0].ins_pack_qstats(slots[:words], cap_e, cap_a)
    assert engs[0].error_flags() == (TABLE_FULL if short == "entry" else ARENA_FULL)
    assert slots[0] == 0 and slots[1] == 0
    slots[words:words + 2] = 0                      # rank 1 sends nothing either
    engs[1].ins_merge_packed_qstats(slots, 2, 1, cap_e, cap_a)
    assert keyed(engs[1]) == before and engs[1].error_flags() == 0


def test_emulated_merge_insertions_with_sums_equals_packed_merge():
    """The host form (merge_insertions with the sums) and the packed form give the same table."""
    b, kw, ref, p = load_fixture("cfg4_ont")
    engs = _sharded(b, kw, 2)
    cap_e, cap_a = _caps(engs)
    slots, _ = _pack_all(engs, cap_e, cap_a)
    ins, qs = engs[0].insertions(), engs[0].qstats()
    engs[1].merge_insertions(ins.sample, ins.pos, ins.count, ins.str_off, ins.chars, qs.ins_rev, qs.ins_qsum, qs.ins_head)
    engs[0].ins_merge_packed_qstats(slots, 2, 0, cap_e, cap_a)
    assert keyed(engs[1]) == keyed(engs[0])


# ---------------------------------------------------------------------------------------------------------------- CPU: gloo
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, name, qstats, out_dir):
    sys.path.insert(0, ROOT); sys.path.insert(0, _HERE)
    import torch.distributed as dist
    import emu_dist_driver
    import test_dist_qstats as m
    emu_dist_driver.install()
    from amplipy_b200 import dist as adist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    b, kw, ref, p = m.load_fixture(name)
    solo = m.emu_engine(kw, qstats)
    ts = solo.process(b, trim=True, pileup=True, qstats=True) if qstats else solo.process(b, trim=True, pileup=True)
    eng = m.emu_engine(kw, qstats)
    t, (first, count) = adist.process_deep_sample(eng, b, qstats=qstats)
    sl = slice(first, first + count)
    assert np.array_equal(t.pos[sl], ts.pos[sl]) and np.array_equal(t.flags[sl], ts.flags[sl])
    assert np.array_equal(eng.counts(), solo.counts())
    assert eng.insertions().as_dict() == solo.insertions().as_dict()
    assert eng.error_flags() == 0
    res = eng.call(ref, p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"], p["min_freq_variants"])
    sres = solo.call(ref, p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"], p["min_freq_variants"])
    assert calling.consensus_string(res, eng.insertions(), 0, p["unknown_symbol"]) == \
        calling.consensus_string(sres, solo.insertions(), 0, p["unknown_symbol"])
    if qstats:
        q, sq = eng.qstats(), solo.qstats()
        assert np.array_equal(q.rev, sq.rev) and np.array_equal(q.qsum, sq.qsum)
        assert m.keyed(eng) == m.keyed(solo)
        rows, cons = m.ivar_outputs(eng, ref, p)
        srows, scons = m.ivar_outputs(solo, ref, p)
        assert len(srows) > 0
        assert "\n".join(rows).encode() == "\n".join(srows).encode()
        assert [c.encode() for c in cons] == [c.encode() for c in scons]
    elif name != "fuzz":
        _, meta, arr = golden_io.load_case(name)
        assert np.array_equal(eng.counts(), arr["counts_aio"]) and eng.insertions().as_dict() == golden_io.ins_from_meta(meta)
    dist.barrier()
    open(os.path.join(out_dir, "ok%d" % rank), "w").write("ok")
    dist.destroy_process_group()


@pytest.mark.parametrize("qstats", [True, False])
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", FIXTURES)
def test_gloo_deep_sample_with_sums(tmp_path, name, world, qstats):
    import torch.multiprocessing as mp
    mp.spawn(_gloo_worker, args=(world, _free_port(), name, qstats, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.isfile(tmp_path / ("ok%d" % r)) for r in range(world))


# ---------------------------------------------------------------------------------------------------------------- GPU
GL = 29903


@pytest.fixture(scope="module")
def stats_oracle():
    d = tempfile.mkdtemp(prefix="amp_xq_test_")
    gcc = "/usr/bin/gcc" if os.path.isfile("/usr/bin/gcc") else "gcc"
    so = os.path.join(d, "libstats_oracle.so")
    subprocess.check_call([gcc, "-O2", "-fPIC", "-shared", "-o", so, os.path.join(_HERE, "stats_oracle.c")])
    olib = ctypes.CDLL(so)
    olib.oracle_pileup_stats_batch.restype = ctypes.c_int64
    yield olib
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture(scope="module")
def gpu_work():
    g = synth.random_genome(GL, 7)
    primers, amps = synth.make_scheme(GL, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    return dict(g=g, tables=find_overlapping_primers(GL, prim, 0), mpl=max_primer_len(prim),
                cfg2=synth.illumina_batch(g, amps, 1_000_000, seed=77, p_ins=0.05), ont=synth.ont_batch(g, amps, 40_000, seed=4))


def _gpu_engine(w, kind, qstats=True):
    from amplipy_b200.engine import Engine
    big = kind == "ont"
    e = Engine(ref_len=GL, primer_tables=w["tables"], max_primer_len=w["mpl"], device=0, ins_slots=(1 << 24) if big else 0,
               ins_arena_bytes=(1 << 30) if big else 0)
    if qstats:
        e.enable_qstats()
    return e


def _gpu_sharded(w, kind, k):
    b = w[kind]
    engs, trims = [], []
    for first, count in read_ranges(b.n, k):
        e = _gpu_engine(w, kind)
        trims.append((first, count, e.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)))
        engs.append(e)
    return engs, trims


def _table_size(e):
    n, nch = ctypes.c_int64(0), ctypes.c_int64(0)
    e.lib.amp_ins_count(e._ctx, ctypes.byref(n), ctypes.byref(nch))
    return int(n.value), int(nch.value)


def _gpu_pack(engs, cap_e, cap_a):
    import torch
    sb = engs[0].ins_slot_bytes_qstats(cap_e, cap_a)
    slots = torch.zeros(sb * len(engs), dtype=torch.uint8, device="cuda:0")
    for r, e in enumerate(engs):
        e.ins_pack_qstats_device(slots.data_ptr() + r * sb, cap_e, cap_a)
    torch.cuda.synchronize()
    return slots, sb


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("kind", ["cfg2", "ont"])
def test_gpu_pack_merge_across_contexts(kind, k, gpu_work, stats_oracle):
    import torch
    from test_ivar import oracle_ins_only_table, oracle_stats
    w = gpu_work
    b = w[kind]
    solo = _gpu_engine(w, kind)
    t = solo.process(b, trim=True, pileup=True, qstats=True)
    want, sq = keyed(solo), solo.qstats()
    assert solo.error_flags() == 0
    engs, trims = _gpu_sharded(w, kind, k)
    assert np.array_equal(sum(e.counts().astype(np.int64) for e in engs), solo.counts())
    assert np.array_equal(sum(e.qstats().rev.astype(np.int64) for e in engs), sq.rev)
    assert np.array_equal(sum(e.qstats().qsum for e in engs), sq.qsum)
    cap_e = max(_table_size(e)[0] for e in engs)
    cap_a = max(_table_size(e)[1] for e in engs)
    slots, sb = _gpu_pack(engs, cap_e, cap_a)
    for r, e in enumerate(engs):
        e.ins_merge_packed_qstats(slots.data_ptr(), k, r, cap_e, cap_a)
    torch.cuda.synchronize()
    for r, e in enumerate(engs):
        assert e.error_flags() == 0
        assert keyed(e) == want, (kind, k, r)
    # and the sums against the serial reference of the pass
    _, _, oins = oracle_stats(stats_oracle, b, GL, 20, {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags})
    got = {(p, s): [rv, q, h] for (_, p, s), (c, rv, q, h) in keyed(engs[-1]).items()}
    assert got == oracle_ins_only_table(oins, got)
    for e in engs + [solo]:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("short", ["entry", "arena"])
def test_gpu_pack_overflow_packs_empty(short, gpu_work):
    import torch
    engs, _ = _gpu_sharded(gpu_work, "cfg2", 2)
    n0, a0 = _table_size(engs[0])
    cap_e, cap_a = (n0 - 1, a0) if short == "entry" else (n0, a0 - 8)
    before = keyed(engs[1])
    sb = engs[0].ins_slot_bytes_qstats(cap_e, cap_a)
    slots = torch.full((2 * sb,), 0xA5, dtype=torch.uint8, device="cuda:0")
    engs[0].ins_pack_qstats_device(slots.data_ptr(), cap_e, cap_a)
    slots[sb:sb + 16] = 0
    engs[1].ins_merge_packed_qstats(slots.data_ptr(), 2, 1, cap_e, cap_a)
    torch.cuda.synchronize()
    assert engs[0].error_flags() == (TABLE_FULL if short == "entry" else ARENA_FULL)
    assert int(slots[:16].count_nonzero()) == 0
    assert keyed(engs[1]) == before and engs[1].error_flags() == 0
    for e in engs:
        e.close()


def _call_bytes(e, g):
    res = e.call(g)
    iv = e.call_ivar(1, 0.03, 0.0)
    ivc = e.call_ivar(10, 0.0, 0.75)
    return [np.ascontiguousarray(getattr(res, f)).tobytes() for f in ("depth", "top_id", "top_count", "pos_flags", "ref_count", "fixed_freq",
                                                                      "fixed_rank", "alt_mask", "ins_freq", "ins_rank", "ins_alt")] + \
        [iv.iupac.tobytes(), iv.fixed_mq.tobytes(), iv.fixed_pval.tobytes(), iv.ins_mq.tobytes(), iv.ins_pval.tobytes(), ivc.iupac.tobytes()]


@pytest.mark.gpu
def test_gpu_one_rank_allreduce_qstats_changes_nothing(gpu_work):
    import torch
    from amplipy_b200.engine import NcclComm
    w = gpu_work
    e = _gpu_engine(w, "cfg2")
    e.process(w["cfg2"].take(np.arange(200_000)), trim=True, pileup=True, qstats=True)
    q0, c0, out0 = e.qstats(), e.counts(), _call_bytes(e, w["g"])
    comm = NcclComm.create(0, 1, 0, NcclComm.unique_id())
    try:
        e.allreduce_qstats(comm)
        torch.cuda.synchronize()
    finally:
        comm.close()
    q1 = e.qstats()
    assert np.array_equal(e.counts(), c0) and np.array_equal(q1.rev, q0.rev) and np.array_equal(q1.qsum, q0.qsum)
    assert _call_bytes(e, w["g"]) == out0
    assert e.error_flags() == 0
    e.close()


@pytest.mark.gpu
def test_gpu_qstats_entry_points_state_errors(gpu_work):
    import torch
    from amplipy_b200.engine import AmpError, NcclComm
    w = gpu_work
    b = w["cfg2"].take(np.arange(20_000))
    plain = _gpu_engine(w, "cfg2", qstats=False)
    assert not plain.qstats_enabled
    plain.process(b, trim=True, pileup=True)
    want = (plain.counts().tobytes(), plain.insertions().as_dict())
    buf = torch.zeros(plain.ins_slot_bytes_qstats(1024, 1 << 16) * 2, dtype=torch.uint8, device="cuda:0")
    comm = NcclComm.create(0, 1, 0, NcclComm.unique_id())
    try:
        with pytest.raises(AmpError):
            plain.allreduce_qstats(comm)                  # refused before NCCL is reached
    finally:
        comm.close()
    with pytest.raises(AmpError):
        plain.ins_pack_qstats_device(buf.data_ptr(), 1024, 1 << 16)
    with pytest.raises(AmpError):
        plain.ins_merge_packed_qstats(buf.data_ptr(), 2, 0, 1024, 1 << 16)
    torch.cuda.synchronize()
    assert (plain.counts().tobytes(), plain.insertions().as_dict()) == want and plain.error_flags() == 0
    st = _gpu_engine(w, "cfg2")
    assert st.qstats_enabled
    st.process(b, trim=True, pileup=True, qstats=True)
    with pytest.raises(AmpError):
        st.allreduce_qstats(0)                            # null communicator
    with pytest.raises(AmpError):
        st.ins_pack_qstats_device(0, 1024, 1 << 16)       # null slot
    with pytest.raises(AmpError):
        st.ins_merge_packed_qstats(0, 2, 0, 1024, 1 << 16)
    assert st.ins_slot_bytes_qstats(-1, 0) == -1 and st.ins_slot_bytes_qstats(3, 20) == 16 + 3 * 32 + 24
    # both contexts stay usable
    for e in (plain, st):
        e.reset()
        e.process(b, trim=True, pileup=True, qstats=e.qstats_enabled)
        assert (e.counts().tobytes(), e.insertions().as_dict()) == want and e.error_flags() == 0
        e.call(w["g"])
    st.call_ivar()
    plain.close(); st.close()


@pytest.mark.gpu
def test_gpu_deep_exchange_chooses_its_form(gpu_work, monkeypatch):
    """A context without the sums: DeepExchange sizes its slots with ins_slot_bytes and calls the existing entry points only,
    and its slot is the one amp_ins_pack_device writes.  A context with them: the *_qstats entry points, and the outputs of a
    one-rank exchange equal those before it."""
    import torch
    import torch.distributed as dist
    from amplipy_b200 import dist as adist
    w = gpu_work
    b = w["cfg2"].take(np.arange(100_000))
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % _free_port(), rank=0, world_size=1)
    try:
        for qstats in (False, True):
            e = _gpu_engine(w, "cfg2", qstats=qstats)
            e.process(b, trim=True, pileup=True, qstats=qstats)
            before = (e.counts().tobytes(), e.insertions().as_dict()) + ((keyed(e), e.qstats().rev.tobytes(), e.qstats().qsum.tobytes())
                                                                        if qstats else ())
            calls = []
            for name in ("allreduce_counts", "ins_pack_device", "ins_merge_packed", "allreduce_qstats", "ins_pack_qstats_device",
                         "ins_merge_packed_qstats"):
                f = getattr(e, name)
                monkeypatch.setattr(e, name, lambda *a, _f=f, _n=name, **k: (calls.append(_n), _f(*a, **k))[1])
            ex = adist.DeepExchange(e, cap_entries=1 << 12, cap_arena_bytes=1 << 18)
            assert ex.qstats == qstats
            if qstats:
                assert ex.slot_bytes == e.ins_slot_bytes_qstats(1 << 12, 1 << 18)
            else:
                assert ex.slot_bytes == e.ins_slot_bytes(1 << 12, 1 << 18) == 16 + 16 * (1 << 12) + (1 << 18)
            ex.run(None)
            torch.cuda.synchronize()
            assert calls == (["allreduce_qstats", "ins_pack_qstats_device", "ins_merge_packed_qstats"] if qstats else
                             ["allreduce_counts", "ins_pack_device", "ins_merge_packed"])
            after = (e.counts().tobytes(), e.insertions().as_dict()) + ((keyed(e), e.qstats().rev.tobytes(), e.qstats().qsum.tobytes())
                                                                       if qstats else ())
            assert after == before and e.error_flags() == 0
            if not qstats:
                ref = torch.zeros_like(ex.send)
                e.lib.amp_ins_pack_device(e._ctx, ctypes.c_void_p(ref.data_ptr()), ctypes.c_int64(1 << 12), ctypes.c_int64(1 << 18), None)
                torch.cuda.synchronize()
                assert torch.equal(ex.send, ref)
            ex.close()
            e.close()
    finally:
        dist.destroy_process_group()
