"""Anchored deletion alleles of the iVar TSV (DESIGN.md 3.7, ``--ivar_deletions``): the table of amp_dels.cuh filled by the strand /
quality pass, its calling, its exchange, the TSV rows and the command line.

CPU: the kernels' own source on the emulator (tests/emu/amp_emu_dels.cpp) against a serial walk of the CIGAR rows written from the
rules of DESIGN.md 3.7 (not from plan_read), p-values against exact arithmetic, rows against a Python build of the rules.
GPU: the same through the C ABI."""
import math
import os
import shutil
import socket
import sys

import numpy as np
import pytest

import emu_dels_driver
import golden_io
import parity
from amplipy_b200 import cli, ivar, synth
from amplipy_b200.batch import ReadBatch
from amplipy_b200.primers import find_overlapping_primers, max_primer_len

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HERE = os.path.join(ROOT, "tests")
DELS_FULL = 128
M, I, D, N, S, H, P, EQ, X = range(9)
F_SKIPPED, F_ERROR = 16, 32
FL = 29903


@pytest.fixture(autouse=True)
def _emulator(monkeypatch):
    emu_dels_driver.install(monkeypatch)


# ---------------------------------------------------------------------------------------------------------------- references
def serial_dels(b, minq, trimmed=None, sample=0):
    """Rule 1 of DESIGN.md 3.7 as a serial walk: {(sample, anchor, len): [count, rev, qsum]}.  ``trimmed``: the trim outputs (pos,
    ncig, flags, cigar rows), whose rows the pileup walked; else the input rows."""
    out = {}
    for i in range(b.n):
        if b.flag[i] & 4:
            continue
        if trimmed is not None:
            if trimmed["flags"][i] & (F_SKIPPED | F_ERROR):
                continue
            a = int(b.cig_off[i]) + 3 * i
            ops = [(int(c & 15), int(c >> 4)) for c in trimmed["cigar"][a:a + int(trimmed["ncig"][i])]]
            r = int(trimmed["pos"][i])
        else:
            ops = b.cigartuples(i)
            r = int(b.pos[i])
        if not ops:
            continue
        qual = b.qual[int(b.qual_off[i]):int(b.qual_off[i + 1])]
        q, prev = 0, None
        for op, n in ops:
            if op == H or n == 0:                 # the walk skips them
                continue
            if op in (M, EQ, X):
                q += n
                r += n
            elif op == D:
                if prev in (M, EQ, X) and int(qual[q - 1]) >= minq:
                    v = out.setdefault((sample, r - 1, n), [0, 0, 0])
                    v[0] += 1
                    v[1] += 1 if b.flag[i] & 16 else 0
                    v[2] += int(qual[q - 1])
                r += n
            elif op == N:
                r += n
            else:                                  # I, S, P advance the query index of the walk
                q += n
            prev = op
    return out


def table(d):
    return {(int(d.sample[k]), int(d.anchor[k]), int(d.len[k])): [int(d.count[k]), int(d.rev[k]), int(d.qsum[k])] for k in range(len(d.count))}


def fisher_exact_less(D, a, mq):
    e = math.floor(D * 10 ** (-mq / 10))
    K, Mt = e + a, 2 * D
    lo, hi = max(0, K - D), min(K, D)
    if e >= hi:
        return 1.0
    return sum(math.comb(K, x) * math.comb(Mt - K, D - x) for x in range(lo, e + 1)) / math.comb(Mt, D)


def fisher_ref(D, a, mq):
    if D <= 2000:
        return fisher_exact_less(D, a, mq)
    from scipy.stats import fisher_exact
    e = math.floor(D * 10 ** (-mq / 10))
    return float(fisher_exact([[e, D - e], [a, D - a]], alternative="less")[1])


def called(want, depth, L, min_depth, min_freq):
    """Rule 4: {key: (mq, pval)} with pval NaN = no row."""
    out = {}
    for (s, a, n), (c, rv, qs) in want.items():
        D = int(depth[s * L + a])
        mq = qs // c if c else 0
        row = D > 0 and D >= min_depth and c and c / D >= min_freq
        out[(s, a, n)] = (mq, fisher_ref(D, c, mq) if row else float("nan"))
    return out


def check_invariant(want, counts_of, L):
    """Rule 3: the events at an anchor never outnumber the bases counted there."""
    at = {}
    for (s, a, n), v in want.items():
        at[(s, a)] = at.get((s, a), 0) + v[0]
    for (s, a), c in at.items():
        assert c <= int(counts_of(s)[:5, a].sum()), (s, a, c)


def emu_engine(kw, slots=0):
    e = emu_dels_driver.EmuDelsEngine(**kw, ins_slots=1 << 18, ins_arena_bytes=1 << 24)
    e.enable_qstats()
    e.enable_dels(slots)
    return e


def trim_dict(t):
    return {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags}


# ---------------------------------------------------------------------------------------------------------------- inputs
def fuzz_inputs():
    g = synth.random_genome(FL, 3)
    primers, amps = synth.make_scheme(FL, 98, seed=4)
    prim = [(s, e) for s, e, _ in primers]
    kw = dict(ref_len=FL, primer_tables=find_overlapping_primers(FL, prim, 0), max_primer_len=max_primer_len(prim))
    return g, amps, kw, {"illumina": synth.illumina_batch(g, amps, 3000, seed=31, p_ins=0.08, p_del=0.08),
                         "ont": synth.ont_batch(g, amps, 150, seed=32, del_rate=0.03)}


def _rec(pos, ops, g, flag=0, q=37, lowq=()):
    """A read whose bases are the reference's where ops align; inserted and clipped bases are 'A'."""
    seq, r = [], pos
    for op, n in ops:
        if op in (M, EQ, X):
            seq.append(g[r:r + n]); r += n
        elif op in (D, N):
            r += n
        elif op in (I, S):
            seq.append("A" * n)
    s = "".join(seq)
    qual = [q] * len(s)
    for j in lowq:
        qual[j] = 5
    return (pos, flag, 0, ops, s, qual)


def hand_batch(g):
    """The shapes of DESIGN.md 3.7 rule 1, forward and reverse; the reads sorted by position."""
    L = len(g)
    recs = [
        _rec(100, [(M, 40), (D, 3), (M, 40)], g),                       # M D M
        _rec(100, [(M, 40), (D, 3), (M, 40)], g, flag=16),
        _rec(110, [(M, 30), (D, 5), (S, 20)], g),                       # M D S
        _rec(120, [(S, 10), (D, 4), (M, 50)], g),                       # S D M: no event
        _rec(130, [(M, 20), (I, 2), (D, 3), (M, 30)], g, flag=16),      # M I D M: no event
        _rec(140, [(M, 20), (N, 50), (M, 30)], g),                      # M N M: no event
        _rec(150, [(M, 25), (D, 2), (N, 10), (M, 30)], g),              # M D N M: the D only
        _rec(160, [(M, 25), (D, 2), (D, 3), (M, 30)], g),               # adjacent D (a read that is not trimmed keeps its row)
        _rec(170, [(M, 25), (D, 2), (M, 30)], g, lowq=(24,)),           # low-quality anchor: no event
        _rec(170, [(M, 25), (D, 2), (M, 30)], g, lowq=(25,)),           # low quality after the deletion: an event
        _rec(0, [(M, 1), (D, 4), (M, 60)], g),                          # deletion right after position 0
        _rec(L - 70, [(M, 60), (D, 10)], g),                            # deletion reaching the last reference base
        _rec(200, [(M, 30), (X, 5), (D, 2), (EQ, 30)], g, flag=16),     # X D =
        _rec(210, [(H, 5), (M, 30), (D, 0), (D, 2), (M, 30)], g),       # an empty op is skipped
    ]
    recs.sort(key=lambda r: r[0])
    return ReadBatch.from_records(recs)


def hand_inputs():
    g = synth.random_genome(FL, 11)
    prim = [(1000, 1020), (5000, 5020)]                                  # no read reaches a primer
    kw = dict(ref_len=FL, primer_tables=find_overlapping_primers(FL, prim, 0), max_primer_len=max_primer_len(prim), min_length=10,
              include_no_primer=True)
    return g, kw, hand_batch(g)


def planted_batch(g, n=2000, at=11287, length=9, frac=0.6, seed=5):
    """n seeded 150-base reads over [at - 100, at + 140), a fraction ``frac`` of them (exactly) carrying a deletion of ``length``
    bases starting at 0-based ``at``; reverse strand for every third read."""
    rng = np.random.default_rng(seed)
    starts = np.sort(rng.integers(at - 100, at - 30, n))
    carry = np.zeros(n, bool)
    carry[rng.permutation(n)[:int(round(frac * n))]] = True
    recs = []
    for i, p in enumerate(starts.tolist()):
        ops = [(M, at - p), (D, length), (M, 150 - (at - p))] if carry[i] else [(M, 150)]
        recs.append(_rec(p, ops, g, flag=16 if i % 3 == 0 else 0, q=int(rng.integers(20, 41))))
    return ReadBatch.from_records(recs)


def _cases():
    return [("golden", n) for n in golden_io.list_cases()] + [("fuzz", "illumina"), ("fuzz", "ont"), ("hand", "hand")]


def load(kind, name):
    if kind == "golden":
        b, meta, arr = golden_io.load_case(name)
        return b, parity.engine_kwargs(meta), bytes(arr["ref_seq"]).decode()
    if kind == "fuzz":
        g, amps, kw, bs = fuzz_inputs()
        return bs[name], kw, g
    g, kw, b = hand_inputs()
    return b, kw, g


# ---------------------------------------------------------------------------------------------------------------- CPU: the table
@pytest.mark.parametrize("trim", [True, False])
@pytest.mark.parametrize("kind,name", _cases())
def test_emulated_table_equals_serial_walk(kind, name, trim):
    b, kw, ref = load(kind, name)
    eng = emu_engine(kw)
    t = eng.process(b, trim=trim, pileup=True, qstats=True)
    want = serial_dels(b, kw.get("min_quality", 20), trim_dict(t) if trim else None)
    got = table(eng.dels())
    assert got == want
    assert (eng.error_flags() & DELS_FULL) == 0
    check_invariant(want, eng.counts, kw["ref_len"])
    if kind == "hand":
        assert (0, 139, 3) in want and (0, 139, 3) in got and want[(0, 139, 3)] == [2, 1, 74]
        assert not any(a in (119, 149) for _, a, _ in want)                    # S D M, M I D M
        assert want[(0, 194, 2)] == [1, 0, 37] and want[(0, 234, 2)] == [1, 1, 37] and (0, 239, 2) in want
        assert (0, 0, 4) in want and (0, FL - 11, 10) in want
        assert (0, 184, 2) in want and (0, 184, 3) not in want              # a D after a D is no event


def test_emulated_pass_without_table_is_unchanged():
    """The strand / quality sums of the pass with the table equal those of the pass without it."""
    b, kw, ref = load("fuzz", "ont")
    a = emu_engine(kw)
    a.process(b, trim=True, pileup=True, qstats=True)
    e = emu_dels_driver.EmuDelsEngine(**kw, ins_slots=1 << 18, ins_arena_bytes=1 << 24)
    e.enable_qstats()
    e.process(b, trim=True, pileup=True, qstats=True)
    qa, qe = a.qstats(), e.qstats()
    assert np.array_equal(qa.rev, qe.rev) and np.array_equal(qa.qsum, qe.qsum) and np.array_equal(qa.ins_qsum, qe.ins_qsum)
    assert np.array_equal(a.counts(), e.counts())


@pytest.mark.parametrize("slots", [1, 2, 64, 1024])
def test_emulated_table_at_full_load(slots):
    """Load factor 1.0 keeps exact sums; one allele more raises DELS_FULL and changes no stored allele; reset clears the table."""
    b, kw, ref = load("hand", "hand")
    eng = emu_engine(kw, slots)
    L = kw["ref_len"]
    # keys whose probes all start on the last slot, so every chain wraps to slot 0
    keys = [(a, n) for a in range(L) for n in (1, 2, 3) if emu_dels_driver.home_slot(a, n, slots) == slots - 1][:slots + 1]
    if len(keys) <= slots:                                                      # too few homed keys: any keys fill the table
        keys = [(a, 1) for a in range(slots + 1)]
    rng = np.random.default_rng(slots)
    vals = [(int(rng.integers(1, 50)), 0, 0) for _ in keys]
    vals = [(c, int(rng.integers(0, c + 1)), int(rng.integers(0, 40 * c))) for c, _, _ in vals]
    d = ivar.Deletions(np.zeros(slots, np.int32), np.array([a for a, _ in keys[:slots]], np.int32), np.array([n for _, n in keys[:slots]], np.int32),
                       *[np.array([v[j] for v in vals[:slots]], dt) for j, dt in ((0, np.int32), (1, np.int32), (2, np.int64))])
    eng.merge_dels(d)
    eng.merge_dels(d)                                                           # every allele found again along its chain
    want = {(0, a, n): [2 * v[0], 2 * v[1], 2 * v[2]] for (a, n), v in zip(keys[:slots], vals)}
    assert table(eng.dels()) == want and eng.error_flags() == 0
    extra = d.take(np.arange(1))
    extra.anchor[:], extra.len[:] = keys[slots][0], keys[slots][1]
    eng.merge_dels(extra)
    assert eng.error_flags() == DELS_FULL
    assert table(eng.dels()) == want
    eng.reset()
    assert len(eng.dels().count) == 0 and eng.error_flags() == 0
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    fresh = emu_engine(kw)
    tf = fresh.process(b, trim=True, pileup=True, qstats=True)
    if len(table(fresh.dels())) <= slots:
        assert table(eng.dels()) == table(fresh.dels()) == serial_dels(b, 20, trim_dict(tf))


def test_emulated_pass_overflow_raises_and_keeps_counts():
    b, kw, ref = load("fuzz", "illumina")
    eng = emu_engine(kw, 64)
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    want = serial_dels(b, 20, trim_dict(t))
    assert len(want) > 64
    assert eng.error_flags() == DELS_FULL
    got = table(eng.dels())
    assert len(got) == 64 and all(got[k][0] <= want[k][0] for k in got)


# ---------------------------------------------------------------------------------------------------------------- CPU: calling and rows
def tsv_with_dels(res, ins, iv, qs, ref_id, ref, counts, want, call, sample=0, L=None, ann=None, names=None):
    """Rules 4-6 built from the rows without the flag: the '-' channel's rows dropped, the anchored deletions with a p-value appended
    after each position's ranked rows in ascending length."""
    L = res.L if L is None else L
    plain = ivar.tsv_rows(res, ins, iv, qs, ref_id, ref, counts, sample, L=L, ann=ann, names=names)
    plain = [r for r in plain if not r[3].startswith("-")]                   # without the flag only the '-' channel's rows start so
    by_pos = {}
    for r in plain:
        by_pos.setdefault(r[1] - 1, []).append(r)
    for (s, a, n), (c, rv, qsum) in sorted(want.items()):
        mq, pv = call[(s, a, n)]
        if s != sample or math.isnan(pv):
            continue
        D = int(res.depth[s * res.L + a])
        rch = "ACGTN".find(ref[a])
        row = (ref_id, a + 1, ref[a], "-" + ref[a + 1:a + 1 + n], int(counts[rch, a]) if rch >= 0 else 0, int(qs.rev[rch, a]) if rch >= 0 else 0,
               int(iv.fixed_mq[s * res.L + a, rch]) if rch >= 0 else 0, c, rv, mq, c / D, D, pv, pv <= ivar.PASS_PVAL)
        cols = ann.columns(sample, a, row[3], names) if ann is not None else ()
        by_pos.setdefault(a, []).extend([row + x for x in cols] if cols else [row])
    return [r for p in sorted(by_pos) for r in by_pos[p]]


@pytest.mark.parametrize("md,mf", [(1, 0.03), (1, 0.0), (20, 0.2)])
@pytest.mark.parametrize("kind,name", [("golden", "cfg2_illumina"), ("golden", "cfg4_ont"), ("fuzz", "ont"), ("hand", "hand")])
def test_emulated_calling_and_rows(kind, name, md, mf):
    b, kw, ref = load(kind, name)
    eng = emu_engine(kw)
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    want = serial_dels(b, kw.get("min_quality", 20), trim_dict(t))
    res = eng.call(ref, 10, 0.0, md, mf)
    d = eng.call_ivar_dels(md, mf)
    call = called(want, res.depth, res.L, md, mf)
    assert table(d) == want
    for k in range(len(d.count)):
        mq, pv = call[(int(d.sample[k]), int(d.anchor[k]), int(d.len[k]))]
        assert int(d.mq[k]) == mq
        assert math.isnan(pv) == math.isnan(d.pval[k])
        if not math.isnan(pv) and pv >= 1e-300:
            assert d.pval[k] == pytest.approx(pv, rel=1e-6, abs=0)
    iv, qs, ins, counts = eng.call_ivar(md, mf), eng.qstats(), eng.insertions(), eng.counts()
    got = ivar.tsv_rows(res, ins, iv, qs, "ref", ref, counts, dels=d)
    exp = tsv_with_dels(res, ins, iv, qs, "ref", ref, counts, want, call)
    assert [r[:12] + r[13:] for r in got] == [r[:12] + r[13:] for r in exp]
    for r, e in zip(got, exp):
        assert r[12] == pytest.approx(e[12], rel=1e-6) or (e[12] < 1e-300 and r[12] < 1e-290)
    assert all((0, r[1] - 1, len(r[3]) - 1) in want for r in got if r[3].startswith("-"))


def test_planted_nine_base_deletion_row():
    g = synth.random_genome(FL, 7)
    b = planted_batch(g)
    kw = dict(ref_len=FL)
    eng = emu_engine(kw)
    eng.process(b, trim=False, pileup=True, qstats=True)
    res = eng.call(g, 10, 0.0, 1, 0.03)
    d = eng.call_ivar_dels(1, 0.03)
    rows = ivar.tsv_rows(res, eng.insertions(), eng.call_ivar(1, 0.03), eng.qstats(), "ref", g, eng.counts(), dels=d)
    drows = [r for r in rows if r[3].startswith("-")]
    assert len(drows) == 1
    r = drows[0]
    assert r[1] == 11287 and r[2] == g[11286] and r[3] == "-" + g[11287:11296]
    assert r[7] == 1200 and r[11] == 2000 and r[10] == 0.6 and r[13]
    plain = ivar.tsv_rows(res, eng.insertions(), eng.call_ivar(1, 0.03), eng.qstats(), "ref", g, eng.counts())
    assert [r[1] for r in plain if r[3].startswith("-")] == list(range(11288, 11297))


def test_pval_body_against_exact():
    lib = emu_dels_driver.lib()
    rng = np.random.default_rng(3)
    for _ in range(200):
        D = int(rng.integers(1, 1500))
        a, mq = int(rng.integers(1, D + 1)), int(rng.integers(0, 45))
        want = fisher_exact_less(D, a, mq)
        if want >= 1e-300:
            assert lib.emu_fisher_less(D, a, mq) == pytest.approx(want, rel=1e-6, abs=0)


# ---------------------------------------------------------------------------------------------------------------- CPU: exchange
def read_ranges(n, k):
    return [(n * r // k, n * (r + 1) // k - n * r // k) for r in range(k)]


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("kind,name", [("golden", "cfg3_deep_alt"), ("golden", "cfg4_ont"), ("fuzz", "illumina")])
def test_emulated_pack_merge_equals_one_context(kind, name, k):
    b, kw, ref = load(kind, name)
    solo = emu_engine(kw)
    solo.process(b, trim=True, pileup=True, qstats=True)
    engs = []
    for first, count in read_ranges(b.n, k):
        e = emu_engine(kw)
        e.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)
        engs.append(e)
    cap = max(len(e.dels().count) for e in engs)
    words = engs[0].dels_slot_bytes(cap) // 8
    slots = np.zeros(k * words, np.uint64)
    for r, e in enumerate(engs):
        e.dels_pack(slots[r * words:(r + 1) * words], cap)
    for r, e in enumerate(engs):
        e.dels_merge_packed(slots, k, r, cap)
        assert table(e.dels()) == table(solo.dels()) and e.error_flags() == 0
    # the host form (merge_dels) gives the same table
    halves = []
    for first, count in read_ranges(b.n, 2):
        e = emu_engine(kw)
        e.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)
        halves.append(e)
    halves[1].merge_dels(halves[0].dels())
    assert table(halves[1].dels()) == table(solo.dels())


def test_emulated_pack_overflow_packs_empty():
    b, kw, ref = load("fuzz", "illumina")
    engs = []
    for first, count in read_ranges(b.n, 2):
        e = emu_engine(kw)
        e.process(b, trim=True, pileup=True, first=first, n=count, qstats=True)
        engs.append(e)
    cap = len(engs[0].dels().count) - 1
    before = table(engs[1].dels())
    words = engs[0].dels_slot_bytes(cap) // 8
    slots = np.full(2 * words, 0xA5A5A5A5A5A5A5A5, np.uint64)
    engs[0].dels_pack(slots[:words], cap)
    assert engs[0].error_flags() == DELS_FULL and slots[0] == 0
    slots[words] = 0
    engs[1].dels_merge_packed(slots, 2, 1, cap)
    assert table(engs[1].dels()) == before and engs[1].error_flags() == 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, kind, name, out_dir):
    sys.path.insert(0, ROOT); sys.path.insert(0, _HERE)
    import torch.distributed as dist
    import emu_dels_driver
    import test_ivar_dels as m
    emu_dels_driver.install()
    from amplipy_b200 import dist as adist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    b, kw, ref = m.load(kind, name)
    solo = m.emu_engine(kw)
    solo.process(b, trim=True, pileup=True, qstats=True)
    eng = m.emu_engine(kw)
    adist.process_deep_sample(eng, b, qstats=True)
    assert m.table(eng.dels()) == m.table(solo.dels()) and eng.error_flags() == 0
    rows = []
    for e in (eng, solo):
        res = e.call(ref, 10, 0.0, 1, 0.03)
        rows.append([ivar.format_row(r) for r in ivar.tsv_rows(res, e.insertions(), e.call_ivar(1, 0.03), e.qstats(), "ref", ref, e.counts(),
                                                               dels=e.call_ivar_dels(1, 0.03))])
    assert len(rows[1]) > 0 and rows[0] == rows[1]
    dist.barrier()
    open(os.path.join(out_dir, "ok%d" % rank), "w").write("ok")
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("kind,name", [("golden", "cfg3_deep_alt"), ("fuzz", "ont")])
def test_gloo_deep_sample_dels(tmp_path, kind, name, world):
    import torch.multiprocessing as mp
    mp.spawn(_gloo_worker, args=(world, _free_port(), kind, name, str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.isfile(tmp_path / ("ok%d" % r)) for r in range(world))


# ---------------------------------------------------------------------------------------------------------------- CPU: command line
GOLD = os.path.join(_HERE, "golden", "cli")


def _run(tmp, tag, cmd, extra):
    j = lambda n: os.path.join(tmp, n)
    for f in ("in.sam", "primers.bed", "ref.fas"):
        if not os.path.isfile(j(f)):
            shutil.copy(os.path.join(GOLD, f), tmp)
    if cmd == "aio":
        cli.main(["aio", "-i", j("in.sam"), "-p", j("primers.bed"), "-r", j("ref.fas"), "-ot", j(tag + ".sam"), "-ov", j(tag + ".vcf"),
                  "-oc", j(tag + ".fas"), "-mfc", "0.2", "-mdc", "3"] + extra)
    else:
        cli.main(["variants", "-i", j("in.sam"), "-r", j("ref.fas"), "-o", j(tag + ".vcf")] + extra)
    return j


def _body(path):
    return [l for l in open(path) if not l.startswith("##source") and not l.startswith("@PG")]


def _cli_reference(j, trim, features=None):
    """The Python build of the deletion rows: the serial walk of the rows the command line's reads were piled up with."""
    from amplipy_b200 import alnio
    from amplipy_b200.primers import load_primers
    ref_id, ref = cli.load_ref_genome(j("ref.fas"))
    L = len(ref)
    b = alnio.read_alignments(j("in.sam")).batch
    prim = load_primers(j("primers.bed"))
    eng = emu_engine(dict(ref_len=L, primer_tables=find_overlapping_primers(L, prim, 0), max_primer_len=max_primer_len(prim)))
    t = eng.process(b, trim=trim, pileup=True, qstats=True)
    want = serial_dels(b, 20, trim_dict(t) if trim else None)
    res = eng.call(ref, 3, 0.2, 1, 0.03)
    ann = names = None
    if features is not None:
        eng.set_features(0, features)
        ann, names = eng.annotate(), [f.name for f in features]
    return tsv_with_dels(res, eng.insertions(), eng.call_ivar(1, 0.03), eng.qstats(), ref_id, ref, eng.counts(), want,
                         called(want, res.depth, L, 1, 0.03), ann=ann, names=names), want


@pytest.mark.parametrize("cmd", ["aio", "variants"])
def test_cli_ivar_deletions(tmp_path, cmd, monkeypatch):
    import amplipy_b200.engine as engine_mod
    monkeypatch.setattr(engine_mod, "Engine", emu_dels_driver.EmuDelsEngine)
    d = str(tmp_path)
    j = _run(d, "plain", cmd, ["--output_tsv", os.path.join(d, "plain.tsv")])
    _run(d, "dels", cmd, ["--output_tsv", j("dels.tsv"), "--ivar_deletions"])
    exts = ("vcf", "sam", "fas") if cmd == "aio" else ("vcf",)
    for ext in exts:
        assert _body(j("dels." + ext)) == _body(j("plain." + ext)), ext
    want_rows, want = _cli_reference(j, cmd == "aio")
    assert any(r[3].startswith("-") and len(r[3]) > 2 for r in want_rows) or len(want) == 0
    got = open(j("dels.tsv")).read().splitlines()
    assert got[0].split("\t") == list(ivar.TSV_HEADER)
    assert len(got) - 1 == len(want_rows)
    for line, r in zip(got[1:], want_rows):
        f, w = line.split("\t"), ivar.format_row(r).split("\t")
        assert f[:12] == w[:12] and f[13:] == w[13:], (f, w)
        assert float(f[12]) == pytest.approx(float(w[12]), rel=1e-6)


def test_cli_ivar_deletions_needs_tsv(tmp_path, monkeypatch):
    import amplipy_b200.engine as engine_mod
    made = []
    monkeypatch.setattr(engine_mod, "Engine", lambda *a, **k: made.append(1))
    with pytest.raises(SystemExit):
        _run(str(tmp_path), "x", "aio", ["--ivar_deletions"])
    with pytest.raises(SystemExit):
        _run(str(tmp_path), "y", "variants", ["--ivar_deletions"])
    assert not made


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu_work():
    g = synth.random_genome(FL, 7)
    primers, amps = synth.make_scheme(FL, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    return dict(g=g, amps=amps, kw=dict(ref_len=FL, primer_tables=find_overlapping_primers(FL, prim, 0), max_primer_len=max_primer_len(prim)),
                cfg2=synth.illumina_batch(g, amps, 1_000_000, seed=1), ont=synth.ont_batch(g, amps, 300_000, seed=4, del_rate=0.03))


def _gpu_engine(w, kind, slots=1 << 22, n_samples=1):
    from amplipy_b200.engine import Engine
    big = kind == "ont"
    e = Engine(**w["kw"], device=0, n_samples=n_samples, ins_slots=(1 << 24) if big else 0, ins_arena_bytes=(1 << 30) if big else 0)
    e.enable_qstats()
    e.enable_dels(slots)
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["cfg2", "ont"])
def test_gpu_table_equals_serial_walk(kind, gpu_work):
    w = gpu_work
    b = w[kind]
    eng = _gpu_engine(w, kind)
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    assert eng.error_flags() == 0
    want = serial_dels(b, 20, trim_dict(t))
    assert table(eng.dels()) == want and len(want) > 100
    check_invariant(want, eng.counts, FL)
    res = eng.call(w["g"])
    d = eng.call_ivar_dels(1, 0.03)
    call = called(want, res.depth, FL, 1, 0.03)
    for k in range(len(d.count)):
        mq, pv = call[(int(d.sample[k]), int(d.anchor[k]), int(d.len[k]))]
        assert int(d.mq[k]) == mq and math.isnan(pv) == math.isnan(d.pval[k])
        if not math.isnan(pv) and pv >= 1e-300:
            assert d.pval[k] == pytest.approx(pv, rel=1e-6, abs=0)
    # halves in reverse order give the same table; reset clears it
    eng.reset()
    assert len(eng.dels().count) == 0
    h = b.n // 2
    eng.process(b, trim=True, pileup=True, qstats=True, first=h, n=b.n - h)
    eng.process(b, trim=True, pileup=True, qstats=True, first=0, n=h)
    assert table(eng.dels()) == want
    eng.reset_async()
    eng.process(b, trim=True, pileup=True, qstats=True)
    assert table(eng.dels()) == want and eng.error_flags() == 0
    eng.close()


@pytest.mark.gpu
def test_gpu_host_device_decoded_paths_agree(gpu_work):
    import tempfile
    from amplipy_b200 import alnio
    w = gpu_work
    b = w["cfg2"].take(np.arange(200_000))
    eng = _gpu_engine(w, "cfg2")
    eng.process(b, trim=True, pileup=True, qstats=True)
    want = table(eng.dels())
    eng.reset()
    eng.process_device(eng.upload(b), trim=True, pileup=True, qstats=True)
    assert table(eng.dels()) == want
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "x.bam")
        alnio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:%d\n" % FL, [("ref", FL)], b)
        raw = open(path, "rb").read()
    eng.reset_async()
    eng.decode_bam(raw, alnio.bam_layout(raw))
    eng.process_decoded(trim=True, pileup=True, qstats=True)
    assert table(eng.dels()) == want and eng.error_flags() == 0


@pytest.mark.gpu
def test_gpu_outputs_unchanged_by_the_table(gpu_work):
    from amplipy_b200.engine import Engine
    w = gpu_work
    b = w["cfg2"].take(np.arange(300_000))
    outs = []
    for dels in (False, True):
        e = Engine(**w["kw"], device=0)
        e.enable_qstats()
        if dels:
            e.enable_dels(1 << 20)
        t = e.process(b, trim=True, pileup=True, qstats=True)
        res = e.call(w["g"])
        q = e.qstats()
        iv = e.call_ivar(1, 0.03)
        outs.append([t.pos.tobytes(), t.flags.tobytes(), t.cigar.tobytes(), e.counts().tobytes(), q.rev.tobytes(), q.qsum.tobytes(),
                     res.depth.tobytes(), iv.fixed_pval.tobytes(), sorted(e.insertions().as_dict().items())])
        e.close()
    assert outs[0] == outs[1]


@pytest.mark.gpu
def test_gpu_plate_spot_checks_solo_runs(gpu_work):
    w = gpu_work
    S = 384
    parts = [w["cfg2"].take(np.arange(k * 2000, (k + 1) * 2000)) for k in range(S)]
    plate = _gpu_engine(w, "cfg2", n_samples=S)
    for s, b in enumerate(parts):
        plate.process(b, trim=True, pileup=True, sample=s, qstats=True)
    assert plate.error_flags() == 0
    allp = table(plate.dels())
    for s in (0, 1, 191, 383):
        solo = _gpu_engine(w, "cfg2", slots=1 << 16)
        solo.process(parts[s], trim=True, pileup=True, qstats=True)
        assert {k: v for k, v in allp.items() if k[0] == s} == {(s,) + k[1:]: v for k, v in table(solo.dels()).items()}
        solo.close()
    plate.close()


@pytest.mark.gpu
def test_gpu_merge_and_packed_exchange(gpu_work):
    import torch
    w = gpu_work
    b = w["ont"].take(np.arange(60_000))
    solo = _gpu_engine(w, "ont")
    solo.process(b, trim=True, pileup=True, qstats=True)
    want = table(solo.dels())
    engs = []
    for first, count in read_ranges(b.n, 2):
        e = _gpu_engine(w, "ont")
        e.process(b, trim=True, pileup=True, qstats=True, first=first, n=count)
        engs.append(e)
    cap = max(len(e.dels().count) for e in engs)
    nb = engs[0].dels_slot_bytes(cap)
    slots = torch.zeros(2 * nb, dtype=torch.uint8, device="cuda:0")
    for r, e in enumerate(engs):
        e.dels_pack_device(slots.data_ptr() + r * nb, cap)
    torch.cuda.synchronize()
    for r, e in enumerate(engs):
        e.dels_merge_packed(slots.data_ptr(), 2, r, cap)
    torch.cuda.synchronize()
    assert all(table(e.dels()) == want and e.error_flags() == 0 for e in engs)
    c = _gpu_engine(w, "ont")
    c.process(b, trim=True, pileup=True, qstats=True, first=0, n=read_ranges(b.n, 2)[0][1])
    f, n = read_ranges(b.n, 2)[1]
    o = _gpu_engine(w, "ont")
    o.process(b, trim=True, pileup=True, qstats=True, first=f, n=n)
    c.merge_dels(o.dels())
    assert table(c.dels()) == want
    small = _gpu_engine(w, "ont")
    small.process(b, trim=True, pileup=True, qstats=True)
    small.dels_pack_device(slots.data_ptr(), cap - 1)
    assert small.error_flags() == DELS_FULL and int(slots[:8].cpu().numpy().view(np.uint64)[0]) == 0


@pytest.mark.gpu
def test_gpu_state_errors(gpu_work):
    from amplipy_b200.engine import AmpError, Engine
    e = Engine(**gpu_work["kw"], device=0)
    with pytest.raises(AmpError):
        e.enable_dels()
    with pytest.raises(AmpError):
        e.dels()
    e.enable_qstats()
    e.enable_dels()
    e.process(gpu_work["cfg2"].take(np.arange(1000)), trim=True, pileup=True, qstats=True)
    with pytest.raises(AmpError):
        e.call_ivar_dels()                     # no amp_call yet
    e.close()


@pytest.mark.gpu
def test_gpu_cli_planted_deletion_and_multi_contig(tmp_path):
    from amplipy_b200 import alnio
    g = synth.random_genome(FL, 7)
    b = planted_batch(g)
    d = str(tmp_path)
    synth.write_fasta(os.path.join(d, "ref.fas"), "ref", g)
    alnio.write_bam(os.path.join(d, "in.bam"), "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:%d\n" % FL, [("ref", FL)], b)
    cli.main(["variants", "-i", os.path.join(d, "in.bam"), "-r", os.path.join(d, "ref.fas"), "-o", os.path.join(d, "v.vcf"),
              "--output_tsv", os.path.join(d, "v.tsv"), "--ivar_deletions"])
    rows = [l.split("\t") for l in open(os.path.join(d, "v.tsv")).read().splitlines()[1:]]
    drows = [r for r in rows if r[3].startswith("-")]
    assert len(drows) == 1 and drows[0][1] == "11287" and drows[0][3] == "-" + g[11287:11296] and float(drows[0][10]) == 0.6
    # two contigs: contig k's rows equal a solo run on its reads
    g2 = synth.random_genome(15000, 8)
    b2 = planted_batch(g2, n=800, at=7000, length=4, frac=0.3, seed=9)
    with open(os.path.join(d, "two.fas"), "w") as f:
        f.write(">ref\n%s\n>seg2\n%s\n" % (g, g2))
    synth.write_fasta(os.path.join(d, "seg2.fas"), "seg2", g2)
    hdr = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:%d\n@SQ\tSN:seg2\tLN:15000\n" % FL
    with open(os.path.join(d, "two.sam"), "w") as f:
        f.write(hdr + "".join(l + "\n" for l in b.sam_lines("ref")) + "".join(l + "\n" for l in b2.sam_lines("seg2")))
    with open(os.path.join(d, "seg2.sam"), "w") as f:
        f.write("@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:seg2\tLN:15000\n" + "".join(l + "\n" for l in b2.sam_lines("seg2")))
    cli.main(["variants", "-i", os.path.join(d, "two.sam"), "-r", os.path.join(d, "two.fas"), "-o", os.path.join(d, "t.vcf"),
              "--output_tsv", os.path.join(d, "t.tsv"), "--ivar_deletions", "--multi_contig"])
    cli.main(["variants", "-i", os.path.join(d, "seg2.sam"), "-r", os.path.join(d, "seg2.fas"), "-o", os.path.join(d, "s.vcf"),
              "--output_tsv", os.path.join(d, "s.tsv"), "--ivar_deletions"])
    two = open(os.path.join(d, "t.tsv")).read().splitlines()
    solo = open(os.path.join(d, "s.tsv")).read().splitlines()
    assert [l for l in two[1:] if l.startswith("seg2\t")] == solo[1:]
    assert any(l.split("\t")[3] == "-" + g2[7000:7004] for l in solo[1:])
