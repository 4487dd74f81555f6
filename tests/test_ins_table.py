"""The insertion-allele table (amp_core.cuh ins_table_add / ins_table_find) at full load, against the oracle.

Reads are built to carry chosen alleles at chosen positions (M, I, M with high qualities), so that the table sees exactly the
distinct keys a case needs: load factor 1.0, every allele on one home slot (the last, so every chain wraps to slot 0), keys
with equal 24-bit tags and different text, keys on both sides of AMP_KEY_SPEC, an arena one record too small, and the
overflow bits.  Inputs are chosen with the device's own hash (emu_driver.ins_hash); the tests never restate it.

CPU: the kernels' own source on the emulator (tests/emu), warp, tile and ONT kernels.
GPU: every producer of the table through the C ABI, with many reads per allele so that slot claims race."""
import os

import numpy as np
import pytest

import emu_driver
import parity
from amplipy_b200 import calling, synth
from amplipy_b200.batch import ReadBatch, pack_seq
from test_ivar import builds  # noqa: F401  (fixture: the iVar emulator and the serial strand / quality reference)

TABLE_FULL, ARENA_FULL, QSTATS_MISS = 16, 32, 64
OP_M, OP_I, OP_D = 0, 1, 2
QUAL = 40
KEY_SPEC = 32          # AMP_KEY_SPEC: keys this long write their arena record before they probe
EL = 3000              # reference length of the emulated cases
SHAPES = {
    # ops before the allele (the last one an M: its last base is the key's anchor), ops after it
    "short": ([(OP_M, 20)], [(OP_M, 20)]),
    "ont": ([(OP_M, 6), (OP_D, 1), (OP_M, 6), (OP_D, 1), (OP_M, 8)], [(OP_M, 8), (OP_D, 1), (OP_M, 6), (OP_D, 1), (OP_M, 6)]),
    "long": ([(OP_M, 600)], [(OP_M, 600)]),
}


def lpad(L):
    return (L + 31) & ~31


def rec_bytes(key):
    """Arena bytes of one record: {int32 gpos, uint32 len} and the text padded to 8 bytes."""
    return 8 * (1 + (len(key) + 7) // 8)


def tag_of(h):
    return (h >> 40) | 0x800000


def _span(ops, consumes):
    return sum(n for op, n in ops if op in consumes)


def make_reads(items, reps=1, shape="short", seed=0, order="shuffle", rev_every=0):
    """A batch with ``reps`` reads per allele; ``items`` = [(pos, key)], key = anchor base + inserted bases (len >= 2).
    order: "shuffle", "round" (allele 0, 1, ..., 0, 1, ...) or "blocks" (all reads of allele 0, then allele 1, ...)."""
    left, right = SHAPES[shape]
    ql, qr = _span(left, (OP_M,)), _span(right, (OP_M,))
    rl = _span(left, (OP_M, OP_D))
    rng = np.random.default_rng(seed)
    idx = np.tile(np.arange(len(items)), reps) if order != "blocks" else np.repeat(np.arange(len(items)), reps)
    if order == "shuffle":
        rng.shuffle(idx)
    pos, cig, seqs, quals, flags = [], [], [], [], []
    for j, i in enumerate(idx):
        p, key = items[i]
        assert len(key) >= 2
        flank = "".join(rng.choice(list("ACGT"), ql - 1 + qr))
        s = flank[:ql - 1] + key + flank[ql - 1:]
        ops = left + [(OP_I, len(key) - 1)] + right
        pos.append(p - rl + 1)
        cig.append([(n << 4) | op for op, n in ops])
        seqs.append(pack_seq(s))
        quals.append(np.full(len(s), QUAL, np.uint8))
        flags.append(16 if rev_every and j % rev_every == 0 else 0)
    n = len(idx)
    off = lambda parts: np.concatenate([[0], np.cumsum([len(x) for x in parts])]).astype(np.uint32)
    cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
    return ReadBatch(np.array(pos, np.int32), np.array(flags, np.uint16), np.zeros(n, np.int32), off(cig), cat(cig, np.uint32),
                     off(seqs), cat(seqs, np.uint8), off(quals), cat(quals, np.uint8))


def random_keys(rng, n, lengths, positions, taken=()):
    """n distinct (pos, key) with pos from ``positions`` and len(key) from ``lengths``."""
    seen, out = set(taken), []
    while len(out) < n:
        it = (int(rng.choice(positions)), "".join(rng.choice(list("ACGT"), int(rng.choice(lengths)))))
        if it not in seen:
            seen.add(it)
            out.append(it)
    return out


def load_items(n, L, seed, margin=30, long_keys=True):
    """n distinct alleles: many at a few positions (more than ten there: call_long_list), the rest spread; lengths 2 .. 40,
    so both sides of AMP_KEY_SPEC, unless long_keys=False."""
    rng = np.random.default_rng(seed)
    lens = list(range(2, 41)) if long_keys else list(range(2, 20))
    crowded = [int(x) for x in rng.choice(np.arange(margin, L - margin), 4, replace=False)]
    spread = np.arange(margin, L - margin)
    k = n // 2
    return random_keys(rng, k, lens, crowded) + random_keys(rng, n - k, lens, spread, [])


def same_home_items(n, mask, L, seed, margin=30, sample=0):
    """n distinct alleles whose hash puts them all on slot ``mask`` (the table's last slot)."""
    rng = np.random.default_rng(seed)
    out, seen = [], set()
    positions = np.arange(margin, L - margin)
    while len(out) < n:
        p = int(rng.choice(positions))
        key = "".join(rng.choice(list("ACGT"), int(rng.integers(2, 12))))
        if (p, key) in seen or emu_driver.ins_hash(sample * lpad(L) + p, key) & mask != mask:
            continue
        seen.add((p, key))
        out.append((p, key))
    return out


_PAIRS = {}


def tag_pairs(length, n_pairs, L, pos=1000, seed=0):
    """Pairs of keys at ``pos`` of the same length and 24-bit tag but different text, whose home slots agree in the lowest
    bit (so that in a two-slot table the second always probes through the first): a birthday search."""
    k = (length, n_pairs, L, pos, seed)
    if k not in _PAIRS:
        rng = np.random.default_rng(1000 + length + seed)
        seen, pairs = {}, []
        for _ in range(200_000):
            key = "".join(rng.choice(list("ACGT"), length))
            h = emu_driver.ins_hash(pos, key)
            t = tag_of(h)
            other = seen.get(t)
            if other is not None and other[0] != key and (other[1] ^ h) & 1 == 0:
                pairs.append((other[0], key))
                del seen[t]
                if len(pairs) == n_pairs:
                    break
            elif other is None:
                seen[t] = (key, h)
        assert len(pairs) == n_pairs, (length, len(pairs))
        _PAIRS[k] = pairs
    return _PAIRS[k]


# ---------------------------------------------------------------------------------------------------------------- checks
def check_calling(res, ins, counts, wc, wins, g, oracle):
    """Depth, consensus, variant records and the rank / frequency of every allele at every position against the oracle."""
    L = len(g)
    ores = oracle.call(wc, wins, g)
    assert np.array_equal(res.depth.astype(np.int64), ores["depth"])
    assert calling.consensus_string(res, ins) == oracle.consensus_string(ores)
    got = calling.variant_records(res, ins, g, counts)
    want = oracle.variant_records(ores, g)
    assert len(got) == len(want)
    for a, c in zip(got, want):
        assert tuple(a[:6]) == tuple(c[:6]) and a[6] == c[6] and a[7] == c[7] and tuple(a[8]) == tuple(c[8]), (a, c)
    arr = {"al_off": ores["al_off"], "al_count": ores["al_count"], "al_freq": ores["al_freq"]}
    meta = {"L": L, "al_sym": [ores["sym"](int(s)) for s in ores["al_sym"][:int(ores["al_off"][L])]]}
    parity.check_allele_order(res, ins, counts, arr, meta)


def check_pileup(eng, b, g, oracle, err=0, call=True, sample=0, trimmed=None, exact=True):
    """Counts, the insertion dict and (call=True) the calling of ``sample`` against the oracle.  err != 0: the table overflowed;
    that bit must be set and every allele that is stored must carry its exact count (exact=False: at most its count, for
    long keys whose later occurrences found the arena full), and some allele must be missing (exact=True)."""
    wc, wins, nerr = oracle.pileup_batch(b, len(g), 20, trimmed=trimmed)
    assert nerr == 0
    assert eng.error_flags() == err
    counts = eng.counts(sample)
    assert np.array_equal(counts.astype(np.int64), wc)
    ins = eng.insertions()
    got = ins.as_dict(sample)
    if err:
        assert all(k in wins and (v == wins[k] if exact else 0 < v <= wins[k]) for k, v in got.items())
        assert len(got) < len(wins) or not exact
        return ins, wins
    assert got == wins
    if call:
        check_calling(eng.call(g), ins, counts, wc, wins, g, oracle)
    return ins, wins


def emu_engine(kernel="v7", **kw):
    kw.setdefault("ins_arena_bytes", 1 << 22)
    return emu_driver.EmuEngine(ref_len=EL, kernel=kernel, **kw)


def emu_chars(eng):
    return int(emu_driver.lib().emu_ins_chars(eng._h))


KERNELS = ["v7", "tile", "ont"]


@pytest.fixture
def emu_ivar(builds, monkeypatch):
    """The emulator build of test_ivar (the strand / quality pass and the iVar calling too) behind emu_driver."""
    monkeypatch.setattr(emu_driver, "lib", lambda: builds[0])


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("nslots", [1, 2, 64, 1024])
@pytest.mark.parametrize("kernel", KERNELS)
def test_load_factor_one(kernel, nslots, oracle_lib):
    g = synth.random_genome(EL, 3)
    items = load_items(nslots + 1, EL, seed=nslots)
    b = make_reads(items[:nslots], reps=3, seed=nslots)
    eng = emu_engine(kernel, ins_slots=nslots)
    eng.process(b, trim=False, pileup=True)
    ins, _ = check_pileup(eng, b, g, oracle_lib)
    assert ins.k == nslots
    # one distinct allele more than the table has slots
    b = make_reads(items, reps=3, seed=nslots + 1)
    eng = emu_engine(kernel, ins_slots=nslots)
    eng.process(b, trim=False, pileup=True)
    ins, _ = check_pileup(eng, b, g, oracle_lib, err=TABLE_FULL)
    assert ins.k == nslots


def test_load_factor_one_aio(oracle_lib):
    """Trim + pileup fused, then calling: reads away from the primers, kept without one (include_no_primer)."""
    g = synth.random_genome(EL, 4)
    prim = [(0, 9), (EL - 10, EL - 1)]
    b = make_reads(load_items(1024, EL, seed=7, margin=100), reps=2, seed=7)
    parity.check_against_oracle(lambda **kw: emu_driver.EmuEngine(kernel="v7", **kw), oracle_lib, b, g, prim, inc=True,
                                ins_slots=1024, arena=1 << 22)


@pytest.mark.parametrize("kernel", KERNELS)
def test_one_home_slot_wraps(kernel, oracle_lib):
    """Every allele hashes to the last slot: the n-th probes n - 1 taken slots, wrapping to slot 0."""
    n = 64
    g = synth.random_genome(EL, 5)
    items = same_home_items(n + 1, n - 1, EL, seed=11)
    for k, err in ((n, 0), (n + 1, TABLE_FULL)):
        b = make_reads(items[:k], reps=4, seed=k, order="round")
        eng = emu_engine(kernel, ins_slots=n)
        eng.process(b, trim=False, pileup=True)
        ins, _ = check_pileup(eng, b, g, oracle_lib, err=err)
        assert ins.k == n


@pytest.mark.parametrize("length", [9, 10, 11, 12, 33])
def test_tag_collisions(length, oracle_lib):
    """Keys with the same gpos, length and tag but other text: the tag matches and the record compare must reject it."""
    g = synth.random_genome(EL, 6)
    pairs = tag_pairs(length, 2, EL)
    for a, c in pairs:
        for first, second in ((a, c), (c, a)):     # each probes through the other
            b = make_reads([(1000, first), (1000, second)], reps=3, order="blocks")
            eng = emu_engine("v7", ins_slots=2)
            eng.process(b, trim=False, pileup=True)
            check_pileup(eng, b, g, oracle_lib)
    # both pairs in one table at load 1.0
    b = make_reads([(1000, k) for pr in pairs for k in pr], reps=3, seed=length)
    eng = emu_engine("v7", ins_slots=4)
    eng.process(b, trim=False, pileup=True)
    check_pileup(eng, b, g, oracle_lib)


@pytest.mark.parametrize("kernel", KERNELS)
def test_key_lengths_around_key_spec(kernel, oracle_lib):
    g = synth.random_genome(EL, 8)
    rng = np.random.default_rng(9)
    items = []
    for n in (KEY_SPEC - 1, KEY_SPEC, KEY_SPEC + 1, 200):
        items += random_keys(rng, 4, [n], [500, 1500], items)
    b = make_reads(items, reps=3, seed=10)
    eng = emu_engine(kernel, ins_slots=16)
    eng.process(b, trim=False, pileup=True)
    check_pileup(eng, b, g, oracle_lib)


@pytest.mark.parametrize("long_keys", [False, True])
def test_arena_one_record_short(long_keys, oracle_lib):
    """An arena that holds every record but the last sets ARENA_FULL, loses that allele alone, and reports no more
    characters than it holds; one record more and everything fits."""
    g = synth.random_genome(EL, 12)
    rng = np.random.default_rng(13)
    lens = [KEY_SPEC, 40, 77] if long_keys else [2, 9, 31]
    items = random_keys(rng, 24, lens, np.arange(100, EL - 100))
    b = make_reads(items, reps=1, seed=14)              # long keys take arena space per occurrence: one each
    need = sum(rec_bytes(k) for _, k in items)
    for arena, err in ((need, 0), (need - 8, ARENA_FULL)):
        eng = emu_engine("v7", ins_slots=32, ins_arena_bytes=arena)
        eng.process(b, trim=False, pileup=True)
        assert emu_chars(eng) <= arena
        ins, _ = check_pileup(eng, b, g, oracle_lib, err=err)
        assert ins.k == len(items) - (1 if err else 0)


def test_long_key_repeats_take_arena_space(oracle_lib):
    """A key of AMP_KEY_SPEC characters or more writes its record before it probes, so every occurrence takes arena space (the
    record of a known allele stays behind unused).  An arena sized for the distinct keys alone then either fits or sets
    ARENA_FULL: counts are never lost without the bit.  Short keys take space once."""
    g = synth.random_genome(EL, 15)
    reps = 6
    for key, arena_recs, err in (("ACGT" * 10, 1, ARENA_FULL), ("ACGT" * 10, reps - 1, ARENA_FULL), ("ACGT" * 10, reps, 0),
                                 ("ACGTACG", 1, 0)):
        b = make_reads([(700, key)], reps=reps, seed=16)
        eng = emu_engine("v7", ins_slots=4, ins_arena_bytes=arena_recs * rec_bytes(key))
        eng.process(b, trim=False, pileup=True)
        check_pileup(eng, b, g, oracle_lib, err=err, exact=False)
        c = eng.insertions().count
        assert (c.sum() == reps) == (err == 0)


@pytest.mark.parametrize("overflow", ["table", "arena"])
def test_reset_after_overflow(overflow, oracle_lib):
    """After an overflow, reset leaves a context whose next run equals a fresh context's, also where the new, shorter keys'
    records land on the stale bytes of the old ones."""
    g = synth.random_genome(EL, 17)
    rng = np.random.default_rng(18)
    old = random_keys(rng, 40, list(range(KEY_SPEC, 60)), [400, 800, 1200])
    new = [(p, k[:len(k) - 1 - i % 7]) for i, (p, k) in enumerate(old[:30])]
    if overflow == "table":
        kw = dict(ins_slots=32, ins_arena_bytes=1 << 20)
    else:
        # room for every occurrence of the new keys (long keys take space per occurrence), not for the old ones
        kw = dict(ins_slots=64, ins_arena_bytes=2 * sum(rec_bytes(k) for _, k in new))
    b_old, b_new = make_reads(old, reps=4, seed=19), make_reads(new, reps=2, seed=20)
    eng = emu_engine("v7", **kw)
    eng.process(b_old, trim=False, pileup=True)
    assert eng.error_flags() == (TABLE_FULL if overflow == "table" else ARENA_FULL)
    eng.reset()
    eng.process(b_new, trim=False, pileup=True)
    fresh = emu_engine("v7", **kw)
    fresh.process(b_new, trim=False, pileup=True)
    check_pileup(eng, b_new, g, oracle_lib)
    assert eng.insertions().as_dict() == fresh.insertions().as_dict()
    r1, r2 = eng.call(g), fresh.call(g)
    for f in ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask"):
        assert np.array_equal(getattr(r1, f), getattr(r2, f)), f


def _tiny_table_class(base):
    from amplipy_b200.engine import AmpError, DEVERR_NAMES

    class TinyTable(base):
        """The engine the CLI makes, with a two-slot insertion table."""

        def __init__(self, **kw):
            kw.update(ins_slots=2, ins_arena_bytes=1 << 16)
            super().__init__(**kw)

        def raise_on_device_errors(self):
            f = self.error_flags()
            if f:
                raise AmpError("; ".join(v for k, v in DEVERR_NAMES.items() if f & k))
    return TinyTable


def _cli_overflow(tmp_path, engine_cls, monkeypatch):
    import shutil
    import amplipy_b200.engine as engine_mod
    from amplipy_b200 import cli
    from amplipy_b200.engine import AmpError
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cli")
    d = str(tmp_path)
    for f in ("in.sam", "primers.bed", "ref.fas"):
        shutil.copy(os.path.join(gold, f), d)
    j = lambda n: os.path.join(d, n)
    monkeypatch.setattr(engine_mod, "Engine", _tiny_table_class(engine_cls))
    outs = [j("out.sam"), j("out.vcf"), j("out.fas"), j("out.tsv")]
    with pytest.raises(AmpError, match="insertion hash table full"):
        cli.main(["aio", "-i", j("in.sam"), "-p", j("primers.bed"), "-r", j("ref.fas"), "-ot", outs[0], "-ov", outs[1], "-oc", outs[2],
                  "--output_tsv", outs[3]])
    assert not any(os.path.exists(p) for p in outs)


def test_cli_table_overflow_writes_nothing(tmp_path, emu_ivar, monkeypatch):
    """aio on an engine whose table overflows: the device error, and no trimmed reads, VCF, TSV or FASTA."""
    from test_ivar import EmuIvarEngine
    _cli_overflow(tmp_path, EmuIvarEngine, monkeypatch)


# ---------------------------------------------------------------------------------------------------------------- GPU
GL = 29903
GPU_REPS = 48          # reads per allele: thousands of occurrences in flight on one slot


@pytest.fixture(scope="module")
def gw():
    """Reference, a primer scheme at the genome's ends, and allele sets for the GPU cases (chosen with the emulator's hash,
    which is the device's: the same header)."""
    g = synth.random_genome(GL, 21)
    return dict(g=g, prim=[(0, 9), (GL - 10, GL - 1)], load=load_items(1024, GL, seed=22, margin=700),
                home=same_home_items(64, 63, GL, seed=23, margin=700))


def gpu_engine(**kw):
    from amplipy_b200.engine import Engine
    kw.setdefault("ins_arena_bytes", 1 << 24)
    return Engine(ref_len=GL, device=0, **kw)


def _oracle_trim(b, prim, w):
    from oracle import oracle
    from amplipy_b200.primers import max_primer_len
    mn, mx = oracle.find_overlapping_primers(GL, prim, 0)
    return oracle.trim_batch(b, GL, mn, mx, max_primer_len(prim), 20, w, 30, True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["warp", "warp_generic", "ont", "tile"])
@pytest.mark.parametrize("items", ["load", "home"])
def test_gpu_producers_at_load_one(case, items, gw, oracle_lib):
    """Every fused kernel at load factor 1.0 (and one allele more: TABLE_FULL, the stored alleles exact)."""
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len
    its = gw[items]
    n = len(its)
    shape = {"warp": "short", "warp_generic": "short", "ont": "ont", "tile": "long"}[case]
    # one home slot: every allele's claim races the others' on the same chain, a thousand occurrences each in flight
    reps = 8 if case == "tile" else 1000 if items == "home" else GPU_REPS
    extra = random_keys(np.random.default_rng(24), 1, [7], [5000], its) if items == "load" else \
        same_home_items(n + 1, n - 1, GL, seed=23, margin=700)[n:]
    for k, err in ((n, 0), (n + 1, TABLE_FULL)):
        b = make_reads((its + extra)[:k], reps=reps, shape=shape, seed=k)
        if case == "warp_generic":          # window width 6: trimming sends every read to the generic phase
            w = 6
            eng = gpu_engine(ins_slots=n, primer_tables=find_overlapping_primers(GL, gw["prim"], 0),
                             max_primer_len=max_primer_len(gw["prim"]), sliding_window_width=w, include_no_primer=True)
            t = eng.process(b, trim=True, pileup=True)
            want = _oracle_trim(b, gw["prim"], w)
            assert np.array_equal(t.flags, want["flags"]) and np.array_equal(t.pos, want["pos"])
            ins, _ = check_pileup(eng, b, gw["g"], oracle_lib, err=err, trimmed=want)
        else:
            eng = gpu_engine(ins_slots=n)
            eng.process(b, trim=False, pileup=True)
            ins, _ = check_pileup(eng, b, gw["g"], oracle_lib, err=err)
        assert ins.k == n
        eng.close()


@pytest.mark.gpu
def test_gpu_entry_points_and_stats_at_load_one(gw, builds, oracle_lib):
    """Host, device and decoded-BAM entry points at load 1.0; the strand / quality pass finds every allele (no bit 64) and its
    sums equal the serial reference."""
    import tempfile
    from amplipy_b200 import alnio
    from test_ivar import oracle_ins_only_table, oracle_stats, stats_dict
    b = make_reads(gw["load"], reps=GPU_REPS, seed=25, rev_every=3)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "x.bam")
        alnio.write_bam(path, "@HD\tVN:1.6\tSO:unsorted\n@SQ\tSN:ref\tLN:%d\n" % GL, [("ref", GL)], b)
        raw = open(path, "rb").read()
    eng = gpu_engine(ins_slots=1024)
    eng.enable_qstats()
    rev, qsum, oins = oracle_stats(builds[1], b, GL, 20)
    for path in ("host", "device", "decoded"):
        if path == "host":
            eng.process(b, trim=False, pileup=True, qstats=True)
        elif path == "device":
            eng.reset_async()
            eng.process_device(eng.upload(b, trim_out=False), trim=False, pileup=True, qstats=True)
        else:
            eng.reset()
            eng.decode_bam(raw, alnio.bam_layout(raw))
            eng.process_decoded(trim=False, pileup=True, qstats=True)
        ins, wins = check_pileup(eng, b, gw["g"], oracle_lib)
        assert ins.k == 1024
        qs = eng.qstats()
        assert np.array_equal(qs.rev.astype(np.int64), rev) and np.array_equal(qs.qsum, qsum)
        assert stats_dict(ins, qs) == oracle_ins_only_table(oins, wins)
        assert eng.error_flags() & QSTATS_MISS == 0
    eng.close()


@pytest.mark.gpu
def test_gpu_plate_and_contigs_share_positions_and_texts(gw, oracle_lib):
    """Two samples with the same positions and texts: distinct gpos, one table at load 1.0; through the plate (a launch per
    sample) and through --multi_contig grouping of interleaved reads."""
    its = gw["load"][:512]
    bs = [make_reads(its, reps=GPU_REPS // 2, seed=26 + s) for s in range(2)]
    plate = gpu_engine(ins_slots=1024, n_samples=2)
    for s, b in enumerate(bs):
        plate.process(b, trim=False, pileup=True, sample=s)
    both = ReadBatch(*[np.concatenate([getattr(bs[0], f), getattr(bs[1], f)[1:] + getattr(bs[0], f)[-1]]) if f.endswith("_off")
                       else np.concatenate([getattr(bs[0], f), getattr(bs[1], f)]) for f in ReadBatch.__dataclass_fields__])
    sid = np.repeat(np.arange(2, dtype=np.int32), bs[0].n)
    perm = np.random.default_rng(27).permutation(both.n)
    contigs = gpu_engine(ins_slots=1024, n_samples=2)
    contigs.process_contigs(both.take(perm), sid[perm], trim=False, pileup=True)
    for eng in (plate, contigs):
        assert eng.insertions().k == 1024
        for s, b in enumerate(bs):
            ins, _ = check_pileup(eng, b, gw["g"], oracle_lib, sample=s, call=False)
        eng.close()


@pytest.mark.gpu
def test_gpu_merge_and_packed_exchange_into_full_table(gw, oracle_lib):
    """merge_insertions and ins_pack_device + ins_merge_packed bring a nearly full table to load 1.0; counts add up."""
    import torch
    its = gw["load"]
    b1 = make_reads(its[:700], reps=GPU_REPS // 2, seed=28)
    b2 = make_reads(its[300:], reps=GPU_REPS // 2, seed=29)
    _, w1, _ = oracle_lib.pileup_batch(b1, GL, 20)
    _, w2, _ = oracle_lib.pileup_batch(b2, GL, 20)
    want = {k: w1.get(k, 0) + w2.get(k, 0) for k in set(w1) | set(w2)}
    assert len(want) == 1024
    a = gpu_engine(ins_slots=1024)
    a.process(b1, trim=False, pileup=True)
    # host merge
    h = gpu_engine(ins_slots=1024)
    h.process(b2, trim=False, pileup=True)
    i1 = a.insertions()
    h.merge_insertions(i1.sample, i1.pos, i1.count, i1.str_off, i1.chars)
    assert h.error_flags() == 0 and h.insertions().as_dict() == want
    # device pack + merge (slot 0: a's table, slot 1: the receiver's own, skipped)
    cap_e, cap_a = 1024, 1 << 24
    sb = a.ins_slot_bytes(cap_e, cap_a)
    slots = torch.zeros(2 * sb // 8, dtype=torch.int64, device="cuda:0")
    a.ins_pack_device(slots.data_ptr(), cap_e, cap_a)
    d = gpu_engine(ins_slots=1024)
    d.process(b2, trim=False, pileup=True)
    d.ins_merge_packed(slots.data_ptr(), 2, 1, cap_e, cap_a)
    torch.cuda.synchronize()
    assert a.error_flags() == 0 and d.error_flags() == 0 and d.insertions().as_dict() == want
    # a slot too small for the table: the bit on the packer, an empty pack, and a merge that changes nothing
    for cap_e2, cap_a2, bit in ((699, cap_a, TABLE_FULL), (cap_e, 64, ARENA_FULL)):
        sb2 = a.ins_slot_bytes(cap_e2, cap_a2)
        small = torch.full((2 * sb2 // 8,), -1, dtype=torch.int64, device="cuda:0")
        p = gpu_engine(ins_slots=1024)
        p.process(b1, trim=False, pileup=True)
        p.ins_pack_device(small.data_ptr(), cap_e2, cap_a2)
        torch.cuda.synchronize()
        assert p.error_flags() == bit
        assert small[0].item() == 0 and small[1].item() == 0
        r = gpu_engine(ins_slots=1024)
        r.process(b2, trim=False, pileup=True)
        before = r.insertions().as_dict()
        r.ins_merge_packed(small.data_ptr(), 2, 1, cap_e2, cap_a2)
        torch.cuda.synchronize()
        assert r.error_flags() == 0 and r.insertions().as_dict() == before
        p.close()
        r.close()
    for e in (a, h, d):
        e.close()


def _ins_count(eng):
    import ctypes
    n, nch = ctypes.c_int64(0), ctypes.c_int64(0)
    assert eng.lib.amp_ins_count(eng._ctx, ctypes.byref(n), ctypes.byref(nch)) == 0
    return int(n.value), int(nch.value)


@pytest.mark.gpu
@pytest.mark.parametrize("long_keys", [False, True])
def test_gpu_export_and_pack_after_arena_full(long_keys, gw, oracle_lib):
    """An arena one record short: ARENA_FULL, n_chars within the arena (checked before anything reads the arena), and the
    export and the pack return exactly the alleles that were stored."""
    import torch
    rng = np.random.default_rng(30)
    lens = [KEY_SPEC, 40, 77] if long_keys else [2, 9, 31]
    items = random_keys(rng, 200, lens, np.arange(700, GL - 700))
    b = make_reads(items, reps=1, seed=31)
    arena = sum(rec_bytes(k) for _, k in items) - 8
    eng = gpu_engine(ins_slots=256, ins_arena_bytes=arena)
    eng.process(b, trim=False, pileup=True)
    n, nch = _ins_count(eng)
    assert nch <= arena, (nch, arena)
    assert eng.error_flags() == ARENA_FULL and n == len(items) - 1
    ins, _ = check_pileup(eng, b, gw["g"], oracle_lib, err=ARENA_FULL)
    got = ins.as_dict()
    sb = eng.ins_slot_bytes(256, arena)
    slots = torch.zeros(2 * sb // 8, dtype=torch.int64, device="cuda:0")
    eng.ins_pack_device(slots.data_ptr(), 256, arena)
    torch.cuda.synchronize()
    assert slots[0].item() == n and slots[1].item() * 8 <= arena
    r = gpu_engine(ins_slots=256)
    r.ins_merge_packed(slots.data_ptr(), 2, 1, 256, arena)
    torch.cuda.synchronize()
    assert r.error_flags() == 0 and r.insertions().as_dict() == got
    eng.close()
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["reset", "reset_async"])
def test_gpu_reset_after_overflow(how, gw, oracle_lib):
    rng = np.random.default_rng(32)
    old = random_keys(rng, 300, list(range(KEY_SPEC, 60)), np.arange(700, 5000))
    new = [(p, k[:len(k) - 1 - i % 7]) for i, (p, k) in enumerate(old[:256])]
    b_old, b_new = make_reads(old, reps=8, seed=33), make_reads(new, reps=8, seed=34)
    eng = gpu_engine(ins_slots=256)
    eng.process(b_old, trim=False, pileup=True)
    assert eng.error_flags() == TABLE_FULL
    getattr(eng, how)()
    eng.process(b_new, trim=False, pileup=True)
    fresh = gpu_engine(ins_slots=256)
    fresh.process(b_new, trim=False, pileup=True)
    check_pileup(eng, b_new, gw["g"], oracle_lib)
    assert eng.insertions().as_dict() == fresh.insertions().as_dict()
    r1, r2 = eng.call(gw["g"]), fresh.call(gw["g"])
    for f in ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask"):
        assert np.array_equal(getattr(r1, f), getattr(r2, f)), f
    eng.close()
    fresh.close()


@pytest.mark.gpu
def test_gpu_cli_table_overflow_writes_nothing(tmp_path, monkeypatch):
    from amplipy_b200.engine import Engine
    _cli_overflow(tmp_path, Engine, monkeypatch)
