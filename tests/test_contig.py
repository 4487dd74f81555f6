"""Multi-contig references (DESIGN.md 3.8): contig k of the FASTA is sample k of one context.

CPU: the grouping source (csrc/amp_contig.cuh) on the emulator (tests/emu/amp_emu_contig.cpp) against numpy -- the plan's totals,
a stable argsort for the permutation, a row gather for the permuted batch, the un-permute and the skipped reads' outputs -- plus
the FASTA / BED / header loaders and the three writers.
GPU: every output of a multi-contig run equals, contig by contig, a single-contig run over that contig's reads, record and BED
rows, for the decoded-BAM and host-array paths, sorted and shuffled input, and through the command line.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from amplipy_b200 import calling, cli, ivar, synth, vcf
from amplipy_b200.batch import ReadBatch
from amplipy_b200.calling import CallResult, Insertions
from amplipy_b200.primers import InputError, load_primers_by_contig

_HERE = os.path.dirname(os.path.abspath(__file__))
TILE, HDR = 2048, 8


def _p(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


@pytest.fixture(scope="module")
def emu():
    d = tempfile.mkdtemp(prefix="amp_contig_test_")
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
    so = os.path.join(d, "libamp_emu_contig.so")
    subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2", "-o", so,
                           os.path.join(_HERE, "emu", "amp_emu_contig.cpp")])
    yield ctypes.CDLL(so)
    shutil.rmtree(d, ignore_errors=True)


def _batch(n, seed):
    recs = synth.fuzz_records(300, n, seed=seed, max_len=40) if n else []
    if not recs:
        z = np.zeros(1, np.uint32)
        return ReadBatch(np.zeros(0, np.int32), np.zeros(0, np.uint16), np.zeros(0, np.int32), z, np.zeros(0, np.uint32), z,
                         np.zeros(0, np.uint8), z, np.zeros(0, np.uint8))
    return ReadBatch.from_records(recs)


def _sids(kind, n, S, rng):
    if kind == "one":
        return np.zeros(n, np.int32)
    if kind == "grouped":                     # contigs in runs, some empty, unmapped reads at the end
        k = np.sort(rng.choice(np.arange(0, S, 2), n))
        k[n - n // 10:] = -1
        return k.astype(np.int32)
    if kind == "interleaved":
        return rng.integers(-1, S, n).astype(np.int32)
    if kind == "runs":                        # contiguous runs, one contig appearing twice
        k = np.repeat(rng.integers(0, S, 6), (n + 5) // 6)[:n]
        return k.astype(np.int32)
    raise ValueError(kind)


def _emu_plan(lib, b, sid, S, nthreads, decoded):
    n = b.n
    table = np.zeros(HDR + 5 * S + (S + 2 if decoded else 0), np.uint64)
    out_sid = np.zeros(max(n, 1), np.int32)
    hist = np.zeros(max((n + TILE - 1) // TILE * S, 1), np.uint32)
    if decoded:                             # records of 8 bytes with the refID at +4; header sequence r = sample r - 1, plus two unknowns
        raw = np.zeros(max(n, 1) * 8, np.uint8)
        rec_off = (np.arange(n, dtype=np.uint64) * 8)
        rid = np.where(sid >= 0, sid + 1, -1).astype(np.int32)
        raw.reshape(-1, 8)[:n, 4:8] = rid.view(np.uint8).reshape(-1, 4)
        r2s = np.array([-2] + list(range(S)) + [-2], np.int32)
        lib.emu_contig_plan(ctypes.c_longlong(n), _p(raw), _p(rec_off), _p(r2s), len(r2s), None, _p(b.flag), _p(b.cig_off), _p(b.qual_off),
                            S, _p(out_sid), _p(hist), _p(table), nthreads)
    else:
        lib.emu_contig_plan(ctypes.c_longlong(n), None, None, None, 0, _p(np.ascontiguousarray(sid)), _p(b.flag), _p(b.cig_off),
                            _p(b.qual_off), S, _p(out_sid), _p(hist), _p(table), nthreads)
    return table, out_sid[:n], hist


def _with_unmapped_flags(b, sid):
    fl = b.flag.copy()
    fl[sid == -1] |= 4
    return ReadBatch(b.pos, fl, b.tlen, b.cig_off, b.cigar, b.seq_off, b.seq, b.qual_off, b.qual)


CASES = [(0, "interleaved", 3), (1, "one", 1), (1, "interleaved", 2), (700, "one", 1), (2047, "grouped", 8), (2048, "interleaved", 5),
         (2049, "runs", 4), (5000, "interleaved", 8), (4100, "grouped", 3), (3000, "interleaved", 40)]


@pytest.mark.parametrize("nthreads", [256, 128, 64])
@pytest.mark.parametrize("n,kind,S", CASES)
def test_emulated_plan_permute_unpermute_match_numpy(n, kind, S, nthreads, emu):
    rng = np.random.default_rng(n * 7 + S)
    sid = _sids(kind, n, S, rng)
    b = _with_unmapped_flags(_batch(n, seed=n + S), sid)
    for decoded in (False, True):
        T, got_sid, hist = _emu_plan(emu, b, sid, S, nthreads, decoded)
        assert np.array_equal(got_sid, sid)
        assert T[2] == 0 and T[0] == (sid == -1).sum()
        ncig = np.diff(b.cig_off.astype(np.int64))
        nq = np.diff(b.qual_off.astype(np.int64))
        assert T[3] == ncig.sum()
        for k in range(S):
            m = sid == k
            assert T[HDR + k] == m.sum()
            assert T[HDR + S + k] == ncig[m].sum() and T[HDR + 2 * S + k] == nq[m].sum()
            if m.any():
                assert int(~np.uint64(T[HDR + 3 * S + k])) == np.flatnonzero(m)[0]
        runs = 1 + int((sid[1:] != sid[:-1]).sum()) if n else 0
        assert T[1] == max(runs - 1, 0)
        present = len(set(sid.tolist()))
        grouped = runs == present
        if grouped:
            for k in range(S):
                if (sid == k).any():
                    assert T[HDR + 4 * S + k] == b.cig_off[np.flatnonzero(sid == k)[0]]
    # stable counting sort + permuted batch
    sel = np.flatnonzero(sid >= 0)
    want_perm = sel[np.argsort(sid[sel], kind="stable")]
    n_in = len(want_perm)
    perm = np.zeros(max(n_in, 1), np.uint32)
    sum_q, sum_s, sum_c = int(b.qual_off[-1]), int(b.seq_off[-1]), int(b.cig_off[-1])
    o = dict(pos=np.zeros(max(n_in, 1), np.int32), flag=np.zeros(max(n_in, 1), np.uint16), tlen=np.zeros(max(n_in, 1), np.int32),
             cig_off=np.zeros(n_in + 1, np.uint32), cigar=np.zeros(sum_c + 1, np.uint32), seq_off=np.zeros(n_in + 1, np.uint32),
             seq=np.zeros(sum_s + 1, np.uint8), qual_off=np.zeros(n_in + 1, np.uint32), qual=np.zeros(sum_q + 1, np.uint8))
    emu.emu_contig_permute(ctypes.c_longlong(n), S, _p(sid), _p(hist), ctypes.c_longlong(n_in), _p(b.pos), _p(b.flag), _p(b.tlen),
                           _p(b.cig_off), _p(b.cigar), _p(b.seq_off), _p(b.seq), _p(b.qual_off), _p(b.qual), _p(perm), _p(o["pos"]),
                           _p(o["flag"]), _p(o["tlen"]), _p(o["cig_off"]), _p(o["cigar"]), _p(o["seq_off"]), _p(o["seq"]),
                           _p(o["qual_off"]), _p(o["qual"]), nthreads)
    assert np.array_equal(perm[:n_in], want_perm)
    wb = b.take(want_perm)
    got = ReadBatch(o["pos"][:n_in], o["flag"][:n_in], o["tlen"][:n_in], o["cig_off"], o["cigar"][:int(o["cig_off"][-1])], o["seq_off"],
                    o["seq"][:int(o["seq_off"][-1])], o["qual_off"], o["qual"][:int(o["qual_off"][-1])])
    for f in ("pos", "flag", "tlen", "cig_off", "cigar", "seq_off", "seq", "qual_off", "qual"):
        assert np.array_equal(getattr(got, f), getattr(wb, f)), f
    # un-permute: rows of the permuted order (at pcig_off[d] + 3d) back to input order (at cig_off[i] + 3i)
    pn = np.diff(o["cig_off"].astype(np.int64))
    po_ncig = np.minimum(pn + rng.integers(0, 4, max(n_in, 1))[:n_in], pn + 3).astype(np.uint16)
    po_cigar = rng.integers(0, 1 << 30, sum_c + 3 * n_in + 1).astype(np.uint32)
    po_pos = rng.integers(0, 1000, max(n_in, 1)).astype(np.int32)
    po_flags = rng.integers(0, 64, max(n_in, 1)).astype(np.uint8)
    out = [np.full(max(n, 1), -7, np.int32), np.zeros(max(n, 1), np.uint16), np.full(max(n, 1), 255, np.uint8),
           np.zeros(sum_c + 3 * n + 1, np.uint32)]
    emu.emu_contig_unpermute(ctypes.c_longlong(n_in), _p(perm), _p(o["cig_off"]), _p(po_pos), _p(po_ncig), _p(po_flags), _p(po_cigar),
                             _p(b.cig_off), _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]), 3, nthreads)
    emu.emu_contig_skip(ctypes.c_longlong(n), _p(sid), _p(b.pos), _p(b.cig_off), _p(b.cigar), _p(out[0]), _p(out[1]), _p(out[2]),
                        _p(out[3]))
    for d, i in enumerate(want_perm.tolist()):
        assert out[0][i] == po_pos[d] and out[1][i] == po_ncig[d] and out[2][i] == po_flags[d]
        a, src = int(b.cig_off[i]) + 3 * i, int(o["cig_off"][d]) + 3 * d
        assert np.array_equal(out[3][a:a + int(po_ncig[d])], po_cigar[src:src + int(po_ncig[d])])
    for i in np.flatnonzero(sid == -1).tolist():      # what the fused kernels write for a read that AmpliPy.py:902 skips
        nc = int(b.cig_off[i + 1] - b.cig_off[i])
        a = int(b.cig_off[i]) + 3 * i
        assert out[0][i] == b.pos[i] and out[1][i] == nc and out[2][i] == 16
        assert np.array_equal(out[3][a:a + nc], b.cigar[b.cig_off[i]:b.cig_off[i + 1]])


def test_emulated_plan_flags_bad_reads(emu):
    b = _batch(50, seed=3)
    fl = b.flag & ~np.uint16(4)
    b = ReadBatch(b.pos, fl, b.tlen, b.cig_off, b.cigar, b.seq_off, b.seq, b.qual_off, b.qual)
    sid = np.zeros(50, np.int32)
    sid[7] = -1                                              # no contig, not flagged unmapped
    T, _, _ = _emu_plan(emu, b, sid, 2, 256, False)
    assert T[2] == 1
    sid[7] = 5                                               # sample id out of range
    T, _, _ = _emu_plan(emu, b, sid, 2, 256, False)
    assert T[2] == 4
    # decoded: header sequence 0 is not in the FASTA; its reads are counted per header sequence
    raw = np.zeros(50 * 8, np.uint8)
    rid = np.where(np.arange(50) < 3, 0, 1).astype(np.int32)
    raw.reshape(-1, 8)[:, 4:8] = rid.view(np.uint8).reshape(-1, 4)
    r2s = np.array([-2, 1], np.int32)
    table = np.zeros(HDR + 5 * 2 + 2, np.uint64)
    emu.emu_contig_plan(ctypes.c_longlong(50), _p(raw), _p(np.arange(50, dtype=np.uint64) * 8), _p(r2s), 2, None, _p(b.flag), _p(b.cig_off),
                        _p(b.qual_off), 2, _p(np.zeros(50, np.int32)), _p(np.zeros(2, np.uint32)), _p(table), 256)
    assert table[2] == 2 and table[HDR + 10] == 3 and table[HDR + 11] == 0 and table[HDR + 1] == 47


# ---------------------------------------------------------------------------------------------------------------- loaders
def test_fasta_loader(tmp_path):
    p = tmp_path / "r.fa"
    p.write_text(">seg1 PB2 segment\nACGT\nAC\n>seg2\nGGGG\nT\n>seg3 x\nN\n")
    assert cli.load_ref_genomes(str(p)) == [("seg1", "ACGTAC"), ("seg2", "GGGGT"), ("seg3", "N")]
    p.write_text(">a\nACGT\n>b\nAC\n>a\nGG\n")
    with pytest.raises(InputError, match="Duplicate"):
        cli.load_ref_genomes(str(p))
    p.write_text(">a\nACGT\n>b\n>c\nGG\n")
    with pytest.raises(InputError, match="Empty sequence"):
        cli.load_ref_genomes(str(p))
    p.write_text(">only\nACGT\nAAA\n")                       # one record: what load_ref_genome reads
    assert cli.load_ref_genomes(str(p)) == [cli.load_ref_genome(str(p))]


def test_bed_by_contig(tmp_path):
    p = tmp_path / "p.bed"
    p.write_text("seg2\t30\t50\tx\nseg1\t10\t20\ty\nseg2\t5\t25\tz\n")
    assert load_primers_by_contig(str(p), ["seg1", "seg2", "seg3"]) == {"seg1": [(10, 20)], "seg2": [(5, 25), (30, 50)], "seg3": []}
    p.write_text("seg1\t10\t20\ty\nsegX\t1\t5\tz\n")
    with pytest.raises(InputError, match="segX"):
        load_primers_by_contig(str(p), ["seg1"])
    p.write_text("seg1\t10\t20\ty\t0\t+\n")                  # 6 columns: rejected like the single-contig loader
    with pytest.raises(InputError, match="Invalid primer BED line"):
        load_primers_by_contig(str(p), ["seg1"])


def test_header_map_and_read_contigs():
    contigs = [("a", "ACGT"), ("b", "ACGTACGT")]
    assert cli.header_contig_map([("b", 8), ("z", 100), ("a", 4)], contigs) == [1, -2, 0]
    with pytest.raises(InputError, match="differs"):
        cli.header_contig_map([("a", 5)], contigs)

    class Aln:
        pass
    aln = Aln()
    aln.refs = [("b", 8), ("z", 100), ("a", 4)]
    aln.sam_fields = [["r0", "0", "a"], ["r1", "4", "*"], ["r2", "0", "b"]]
    aln.n = 3
    assert cli.sam_read_contigs(aln, contigs).tolist() == [0, -1, 1]   # an unknown header sequence without reads is fine
    aln.sam_fields.append(["r3", "0", "z"])
    aln.n = 4
    with pytest.raises(InputError, match=": z"):
        cli.sam_read_contigs(aln, contigs)
    aln.refs = []                                                     # no @SQ lines: RNAME names the FASTA record
    aln.sam_fields = [["r0", "0", "b"], ["r1", "0", "a"]]
    aln.n = 2
    assert cli.sam_read_contigs(aln, contigs).tolist() == [1, 0]


def test_check_contig_plan_messages():
    from amplipy_b200.engine import ContigPlan
    plan = ContigPlan(2, 3)
    plan.c.errors = 2
    plan.ref_reads[:] = [0, 5, 0]
    with pytest.raises(InputError, match="not in the reference FASTA: y"):
        cli.check_contig_plan(plan, [("x", 1), ("y", 2), ("w", 3)], [-2, -2, 0])
    plan.c.errors = 1
    with pytest.raises(InputError, match="flag 4"):
        cli.check_contig_plan(plan)
    plan.c.errors = 0
    cli.check_contig_plan(plan)


# ---------------------------------------------------------------------------------------------------------------- writers
def _call_result(L, S, rng):
    SL = S * L
    top = rng.integers(-1, 6, SL).astype(np.int32)
    flags = rng.integers(0, 8, SL).astype(np.uint8)
    freq = rng.random((SL, 6))
    rank = np.tile(np.arange(6, dtype=np.int32), (SL, 1))
    alt = rng.integers(0, 64, SL).astype(np.uint8)
    return CallResult(L, S, rng.integers(1, 100, SL).astype(np.int32), top, np.ones(SL, np.int32), flags,
                      rng.integers(0, 50, SL).astype(np.int32), freq, rank, alt, np.zeros(1), np.zeros(1, np.int32), np.zeros(1, np.uint8))


def test_writers_take_a_contig_length():
    rng = np.random.default_rng(5)
    L, lens = 40, [40, 23]
    res = _call_result(L, 2, rng)
    ins = Insertions(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), [])
    seqs = ["".join(rng.choice(list("ACGT"), n)) for n in lens]
    counts = [rng.integers(0, 9, (6, L)).astype(np.int32) for _ in lens]
    # one sample cut to its contig's length = the same sample in a context of that length
    for k, n in enumerate(lens):
        solo = CallResult(n, 1, *[getattr(res, f)[k * L:k * L + n] for f in ("depth", "top_id", "top_count", "pos_flags", "ref_count",
                                                                                  "fixed_freq", "fixed_rank", "alt_mask")],
                          res.ins_freq, res.ins_rank, res.ins_alt)
        cons = calling.consensus_string(res, ins, k, "N", L=n)
        assert len(cons) == n and cons == calling.consensus_string(solo, ins, 0, "N")
        assert calling.variant_records(res, ins, seqs[k], counts[k], k, L=n) == calling.variant_records(solo, ins, seqs[k], counts[k][:, :n])
    recs = [calling.variant_records(res, ins, seqs[k], counts[k], k, L=n) for k, n in enumerate(lens)]
    assert recs[0] and recs[1]
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.vcf")
        vcf.write_vcf(path, ["seg1", "seg2"], "0.0.2", ["prog"], recs)
        lines = open(path).read().splitlines()
    assert [l for l in lines if l.startswith("##contig")] == ["##contig=<ID=seg1>", "##contig=<ID=seg2>"]
    body = [l for l in lines if not l.startswith("#")]
    assert body == [vcf.record_line("seg1", r) for r in recs[0]] + [vcf.record_line("seg2", r) for r in recs[1]]
    assert vcf.header_text(["seg1"], "v", ["p"]) == vcf.header_text("seg1", "v", ["p"])
    # TSV: REGION is the contig's ID, positions within its length
    pv = np.full((2 * L, 6), np.nan)
    pv[3, 1] = 0.01
    pv[L + 20, 2] = 0.2
    pv[L + 30, 2] = 0.3                                   # past contig 2's end: cut
    iv = ivar.IvarResult(np.zeros(2 * L, np.uint8), np.full((2 * L, 6), 30, np.int32), pv, np.zeros(1, np.int32), np.full(1, np.nan))
    qs = ivar.QStats(np.zeros((6, L), np.int32), np.zeros((6, L), np.int64), np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.uint8))
    r1 = ivar.tsv_rows(res, ins, iv, qs, "seg1", seqs[0], counts[0], 0, L=40)
    r2 = ivar.tsv_rows(res, ins, iv, qs, "seg2", seqs[1], counts[1], 1, L=23)
    assert [(r[0], r[1]) for r in r1] == [("seg1", 4)] and [(r[0], r[1]) for r in r2] == [("seg2", 21)]


# ---------------------------------------------------------------------------------------------------------------- GPU
SEG_LENS = [2341, 2341, 2233, 1778, 1565, 1413, 1027, 890]     # influenza-A-like segment lengths
SEG_IDS = ["seg%d" % (k + 1) for k in range(8)]


@pytest.fixture(scope="module")
def segs():
    out = []
    for k, L in enumerate(SEG_LENS):
        g = synth.random_genome(L, 100 + k)
        primers, amps = synth.make_scheme(L, max(2, (L - 60) // 260), amp_len=300, seed=10 + k)
        prim = sorted((s, e) for s, e, _ in primers)
        b = synth.illumina_batch(g, amps, 6000 + 1500 * k, seed=20 + k, snvs=[(L // 3, "ACGT"[k % 4], 0.4)])
        if k == 2:                                               # a few ONT-like reads on one contig
            b = ReadBatch.concat([b, synth.ont_batch(g, amps, 300, seed=30)])
        out.append(dict(id=SEG_IDS[k], g=g, L=L, primers=primers, prim=prim, b=b))
    return out


def _solo(seg, trim=True, qstats=True):
    from amplipy_b200.engine import Engine
    from amplipy_b200.primers import find_overlapping_primers, max_primer_len
    L = seg["L"]
    e = Engine(ref_len=L, primer_tables=find_overlapping_primers(L, seg["prim"], 0), max_primer_len=max_primer_len(seg["prim"]),
               ins_slots=1 << 20, ins_arena_bytes=1 << 26)
    e.enable_qstats()
    t = e.process(seg["b"], trim=trim, pileup=True, qstats=qstats)
    return e, t


def _multi_engine(segs, ins_slots=1 << 20, ins_arena_bytes=1 << 26):
    from amplipy_b200.engine import Engine
    e = Engine(ref_len=max(s["L"] for s in segs), n_samples=len(segs), ins_slots=ins_slots, ins_arena_bytes=ins_arena_bytes)
    for k, s in enumerate(segs):
        e.set_scheme(k, s["prim"], 0, ref_len=s["L"])
        e.set_sample_reference(k, s["g"])
    e.enable_qstats()
    return e


def _combined(segs, n_unmapped=37, seed=0):
    """The contigs' batches one after another (grouped) with unmapped reads at the end, and their sample ids."""
    rng = np.random.default_rng(seed)
    extra = segs[0]["b"].take(rng.choice(segs[0]["b"].n, n_unmapped, replace=False))
    extra = ReadBatch(extra.pos, extra.flag | np.uint16(4), extra.tlen, extra.cig_off, extra.cigar, extra.seq_off, extra.seq,
                      extra.qual_off, extra.qual)
    b = ReadBatch.concat([s["b"] for s in segs] + [extra])
    sid = np.concatenate([np.full(s["b"].n, k, np.int32) for k, s in enumerate(segs)] + [np.full(n_unmapped, -1, np.int32)])
    return b, sid


def _ins_key_dict(ins, values, sample):
    return {(int(ins.pos[j]), ins.strs[j]): v for j, v in enumerate(values) if ins.sample[j] == sample}


def _check_against_solo(multi, segs, t, sid, order, trim, qstats=True, ivar_too=True):
    """Everything multi computed for contig k == a solo run over contig k's reads (``order``: multi's read i is batch row order[i])."""
    res = multi.call(None)
    mins = multi.insertions()
    Lm = multi.L
    ivs = [multi.call_ivar(1, 0.03, 0.0), multi.call_ivar(10, 0.0, 0.7)] if ivar_too else []
    starts = np.concatenate([[0], np.cumsum([s["b"].n for s in segs])])
    for k, seg in enumerate(segs):
        L = seg["L"]
        solo, st = _solo(seg, trim=trim, qstats=qstats)
        if trim:
            rows = np.flatnonzero(sid == k)                       # multi's reads of contig k, in multi's order
            src = order[rows] - starts[k]
            assert np.array_equal(t.pos[rows], st.pos[src]) and np.array_equal(t.ncig[rows], st.ncig[src])
            assert np.array_equal(t.flags[rows], st.flags[src])
            for i, j in zip(rows[::97].tolist(), src[::97].tolist()):
                assert t.cigartuples(i) == st.cigartuples(j)
        c = multi.counts(k)
        assert np.array_equal(c[:, :L], solo.counts()) and not c[:, L:].any()
        sins = solo.insertions()
        assert _ins_key_dict(mins, mins.count.tolist(), k) == sins.as_dict()
        sres = solo.call(seg["g"])
        sl = slice(k * Lm, k * Lm + L)
        for f in ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask"):
            assert getattr(res, f)[sl].tobytes() == getattr(sres, f).tobytes(), f
        tm, ts = res.top_id[sl], sres.top_id
        assert np.array_equal(tm[ts < 6], ts[ts < 6])
        assert [mins.strs[x - 6] for x in tm[ts >= 6]] == [sins.strs[x - 6] for x in ts[ts >= 6]]
        for f in ("ins_freq", "ins_rank", "ins_alt"):
            assert _ins_key_dict(mins, getattr(res, f)[:mins.k].tolist(), k) == _ins_key_dict(sins, getattr(sres, f)[:sins.k].tolist(), 0), f
        if qstats:
            q, sq = multi.qstats(k), solo.qstats(0)
            assert np.array_equal(q.rev[:, :L], sq.rev) and np.array_equal(q.qsum[:, :L], sq.qsum)
            for f in ("ins_rev", "ins_qsum", "ins_head"):
                assert _ins_key_dict(mins, getattr(q, f).tolist(), k) == _ins_key_dict(sins, getattr(sq, f).tolist(), 0), f
        for (mdp, mf, th), iv in zip(((1, 0.03, 0.0), (10, 0.0, 0.7)), ivs):
            siv = solo.call_ivar(mdp, mf, th)
            assert iv.iupac[sl].tobytes() == siv.iupac.tobytes() and iv.fixed_mq[sl].tobytes() == siv.fixed_mq.tobytes()
            assert iv.fixed_pval[sl].tobytes() == siv.fixed_pval.tobytes()
            assert _ins_key_dict(mins, iv.ins_mq[:mins.k].tolist(), k) == _ins_key_dict(sins, siv.ins_mq[:sins.k].tolist(), 0)
            assert (np.array(list(_ins_key_dict(mins, iv.ins_pval[:mins.k].tolist(), k).values())).tobytes() ==
                    np.array([dict(_ins_key_dict(sins, siv.ins_pval[:sins.k].tolist(), 0))[key]
                              for key in _ins_key_dict(mins, iv.ins_pval[:mins.k].tolist(), k)]).tobytes())
        solo.close()
    if trim:
        un = np.flatnonzero(sid == -1)
        assert (t.flags[un] == 16).all()
    assert multi.error_flags() == 0


def _write_multi_bam(path, b, sid, segs, names=None):
    from amplipy_b200 import alnio
    hdr = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (s["id"], s["L"]) for s in segs) + \
          "@PG\tID:synth\tPN:synth\tVN:1\n"
    alnio.write_bam(path, hdr, [(s["id"], s["L"]) for s in segs], b, names=names, refid=sid)
    return hdr


@pytest.mark.gpu
@pytest.mark.parametrize("trim", [True, False])
@pytest.mark.parametrize("shuffled", [False, True])
def test_gpu_host_arrays_equal_single_contig_runs(segs, trim, shuffled):
    b, sid = _combined(segs)
    order = np.random.default_rng(1).permutation(b.n) if shuffled else np.arange(b.n)
    bb, ss = b.take(order), sid[order]
    multi = _multi_engine(segs)
    t = multi.process_contigs(bb, ss, trim=trim, pileup=True, qstats=True)
    assert multi.contig_plan.grouped == (not shuffled)
    _check_against_solo(multi, segs, t, ss, order, trim)


@pytest.mark.gpu
@pytest.mark.parametrize("shuffled", [False, True])
def test_gpu_decoded_bam_equals_single_contig_runs(segs, shuffled):
    from amplipy_b200 import alnio
    from amplipy_b200.engine import TrimResult
    b, sid = _combined(segs)
    order = np.random.default_rng(2).permutation(b.n) if shuffled else np.arange(b.n)
    bb, ss = b.take(order), sid[order]
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "x.bam")
        # header order differs from the FASTA's: the map goes by name
        segs_rev = segs[::-1]
        rid = np.where(ss >= 0, len(segs) - 1 - ss, -1).astype(np.int32)
        _write_multi_bam(path, bb, rid, segs_rev)
        raw = open(path, "rb").read()
    layout = alnio.bam_layout(raw)
    multi = _multi_engine(segs)
    multi.decode_bam(raw, layout)
    plan = multi.contig_plan_decoded(cli.header_contig_map(layout["refs"], [(s["id"], s["g"]) for s in segs]))
    assert plan.errors == 0 and plan.grouped == (not shuffled) and plan.n_no_contig == (ss == -1).sum()
    assert plan.reads.tolist() == [int((ss == k).sum()) for k in range(len(segs))]
    outs = multi.process_decoded_contigs(trim=True, pileup=True, qstats=True)
    db, _ = multi.decoded_batch()
    _check_against_solo(multi, segs, TrimResult(db, *outs), ss, order, True)


@pytest.mark.gpu
def test_gpu_read_past_contig_end_raises_coordinate_error(segs):
    from amplipy_b200.engine import AmpError
    two = [segs[0], segs[7]]                                          # 2341 and 890 bases: the context is 2341 long
    b, sid = _combined(two, n_unmapped=0)
    pos = b.pos.copy()
    pos[np.flatnonzero(sid == 1)[0]] = two[1]["L"] - 5                # runs past the short contig's end, not past the context's
    bad = ReadBatch(pos, b.flag & ~np.uint16(4), b.tlen, b.cig_off, b.cigar, b.seq_off, b.seq, b.qual_off, b.qual)
    multi = _multi_engine(two)
    multi.process_contigs(bad, sid, trim=False, pileup=True)
    assert multi.error_flags() & 1
    with pytest.raises(AmpError, match="outside the reference"):
        multi.raise_on_device_errors()
    ok = _multi_engine(two)
    ok.process_contigs(b, sid, trim=False, pileup=True)
    assert ok.error_flags() == 0
    with pytest.raises(AmpError):                                      # refID -1 without flag 4
        _multi_engine(two).process_contigs(bad, np.full(bad.n, -1, np.int32), trim=False, pileup=True)


@pytest.mark.gpu
def test_gpu_one_million_reads_sorted_equals_shuffled(segs):
    reps = [dict(s, b=synth.illumina_batch(s["g"], synth.make_scheme(s["L"], max(2, (s["L"] - 60) // 260), amp_len=300, seed=10 + k)[1],
                                           125_000, seed=50 + k)) for k, s in enumerate(segs)]
    b, sid = _combined(reps, n_unmapped=100)
    order = np.random.default_rng(3).permutation(b.n)
    outs = []
    for o in (np.arange(b.n), order):
        m = _multi_engine(segs, ins_slots=1 << 22, ins_arena_bytes=1 << 28)
        t = m.process_contigs(b.take(o), sid[o], trim=True, pileup=True, qstats=True)
        inv = np.empty_like(o)
        inv[o] = np.arange(b.n)
        res = m.call(None)
        ins = m.insertions()
        q = [m.qstats(k) for k in range(len(segs))]
        outs.append(dict(pos=t.pos[inv], ncig=t.ncig[inv], flags=t.flags[inv], counts=[m.counts(k) for k in range(len(segs))],
                         ins={(int(s_), int(p_), st): int(c_) for s_, p_, c_, st in zip(ins.sample, ins.pos, ins.count, ins.strs)},
                         res=[getattr(res, f).tobytes() for f in ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank",
                                                                  "alt_mask")],
                         q=[(x.rev.tobytes(), x.qsum.tobytes()) for x in q], grouped=m.contig_plan.grouped))
        assert m.error_flags() == 0
        m.close()
    a, c = outs
    assert a["grouped"] and not c["grouped"]
    for f in ("pos", "ncig", "flags"):
        assert np.array_equal(a[f], c[f]), f
    assert all(np.array_equal(x, y) for x, y in zip(a["counts"], c["counts"]))
    assert a["ins"] == c["ins"] and a["res"] == c["res"] and a["q"] == c["q"]


# ---- the command line
def _split_inputs(d, segs, b, sid, fmt):
    """The multi-contig FASTA / BED / reads, and per contig the single-contig FASTA / BED / reads."""
    from amplipy_b200 import alnio
    j = lambda n: os.path.join(d, n)
    with open(j("multi.fas"), "w") as f:
        for s in segs:
            f.write(">%s some description\n" % s["id"])
            for i in range(0, s["L"], 60):
                f.write(s["g"][i:i + 60] + "\n")
    with open(j("multi.bed"), "w") as f:
        for s in segs[::-1]:
            for st, en, nm in s["primers"]:
                f.write("%s\t%d\t%d\t%s\n" % (s["id"], st, en, nm))
    names = ["q%d" % i for i in range(b.n)]
    hdr = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (s["id"], s["L"]) for s in segs) + "@PG\tID:synth\tPN:synth\tVN:1\n"
    if fmt == "bam":
        alnio.write_bam(j("multi.bam"), hdr, [(s["id"], s["L"]) for s in segs], b, names=names, refid=sid)
    else:
        lines = []
        for i in range(b.n):
            rn = segs[sid[i]]["id"] if sid[i] >= 0 else "*"
            lines.append(b.take(np.array([i])).sam_lines(rname=rn, name_prefix="x")[0].replace("x0", names[i], 1))
        with open(j("multi.sam"), "w") as f:
            f.write(hdr + "\n".join(lines) + "\n")
    for k, s in enumerate(segs):
        synth.write_fasta(j("%s.fas" % s["id"]), s["id"], s["g"])
        synth.write_bed(j("%s.bed" % s["id"]), s["primers"], rname=s["id"])
        sel = np.flatnonzero(sid == k)
        h = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:%s\tLN:%d\n@PG\tID:synth\tPN:synth\tVN:1\n" % (s["id"], s["L"])
        if fmt == "bam":
            alnio.write_bam(j("%s.bam" % s["id"]), h, [(s["id"], s["L"])], b.take(sel), names=[names[i] for i in sel])
        else:
            with open(j("%s.sam" % s["id"]), "w") as f:
                f.write(h + "\n".join(lines[i] for i in sel) + "\n")
    return j


def _body(path, skip="#"):
    return [l for l in open(path).read().splitlines() if not l.startswith(skip)]


def _records(path):
    from amplipy_b200 import alnio
    a = alnio.read_alignments(path)
    return [(a.batch.record(i)[:2], a.batch.record(i)[3]) for i in range(a.n)], a


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bam", "sam"])
def test_gpu_cli_aio_equals_per_contig_runs(tmp_path, segs, fmt):
    small = [dict(s, b=s["b"].take(np.arange(min(s["b"].n, 3000)))) for s in segs]
    b, sid = _combined(small, n_unmapped=11)
    d = str(tmp_path)
    j = _split_inputs(d, small, b, sid, fmt)
    opts = ["-mdc", "3", "--iupac_threshold", "0.6"]
    cli.main(["aio", "--multi_contig", "-i", j("multi." + fmt), "-p", j("multi.bed"), "-r", j("multi.fas"), "-ot", j("m_trim." + fmt),
              "-ov", j("m.vcf"), "-oc", j("m.fas"), "--output_tsv", j("m.tsv")] + opts)
    vcf_rows, tsv_rows, cons, trimmed = [], [], [], []
    for s in small:
        p = s["id"]
        cli.main(["aio", "-i", j(p + "." + fmt), "-p", j(p + ".bed"), "-r", j(p + ".fas"), "-ot", j(p + "_trim." + fmt), "-ov", j(p + ".vcf"),
                  "-oc", j(p + "_c.fas"), "--output_tsv", j(p + ".tsv")] + opts)
        vcf_rows += _body(j(p + ".vcf"))
        tsv_rows += _body(j(p + ".tsv"), "REGION")
        cons.append(">%s\n%s\n" % (p, open(j(p + "_c.fas")).read().split("\n")[1]))
        trimmed += _records(j(p + "_trim." + fmt))[0]
    assert _body(j("m.vcf")) == vcf_rows and len(vcf_rows) > 0
    assert [l for l in open(j("m.vcf")) if l.startswith("##contig")] == ["##contig=<ID=%s>\n" % s["id"] for s in small]
    assert _body(j("m.tsv"), "REGION") == tsv_rows and len(tsv_rows) > 0
    assert open(j("m.fas")).read() == "".join(cons)
    got, _ = _records(j("m_trim." + fmt))
    assert got == trimmed
    # trim, then variants / consensus on the trimmed file == the same steps per contig (aio piles up the reads the trim step drops
    # for length, as AmpliPy.py does, so the steps are compared with the steps)
    steps = ["variants", "-o", "{o}.vcf", "--output_tsv", "{o}.tsv"], ["consensus", "-o", "{o}.fas", "-md", "3", "--iupac_threshold", "0.6"]

    def pipeline(tag, inp, bed, fas, extra):
        cli.main(["trim"] + extra + ["-i", inp, "-p", bed, "-r", fas, "-o", j(tag + "_t." + fmt)])
        for st in steps:
            cli.main([st[0]] + extra + ["-i", j(tag + "_t." + fmt), "-r", fas] + [x.format(o=j(tag)) for x in st[1:]])
    pipeline("s", j("multi." + fmt), j("multi.bed"), j("multi.fas"), ["--multi_contig"])
    assert _records(j("s_t." + fmt))[0] == got
    want_v, want_t, want_c = [], [], []
    for s in small:
        p = s["id"]
        pipeline("p" + p, j(p + "." + fmt), j(p + ".bed"), j(p + ".fas"), [])
        want_v += _body(j("p%s.vcf" % p))
        want_t += _body(j("p%s.tsv" % p), "REGION")
        want_c.append(">%s\n%s\n" % (p, open(j("p%s.fas" % p)).read().split("\n")[1]))
    assert _body(j("s.vcf")) == want_v and _body(j("s.tsv"), "REGION") == want_t and open(j("s.fas")).read() == "".join(want_c)


@pytest.mark.gpu
def test_gpu_cli_single_record_fasta_unchanged_by_the_flag(tmp_path, segs):
    s = dict(segs[0], b=segs[0]["b"].take(np.arange(4000)))
    d = str(tmp_path)
    j = _split_inputs(d, [s], s["b"], np.zeros(s["b"].n, np.int32), "bam")
    p = s["id"]
    outs = {}
    for tag, extra in (("plain", []), ("flag", ["--multi_contig"])):
        cli.main(["aio", "-i", j(p + ".bam"), "-p", j(p + ".bed"), "-r", j(p + ".fas"), "-ot", j(tag + ".bam"), "-ov", j(tag + ".vcf"),
                  "-oc", j(tag + ".fas"), "--output_tsv", j(tag + ".tsv")] + extra)
        recs, aln = _records(j(tag + ".bam"))                          # the @PG line records the command line, flag included
        outs[tag] = [recs, [l for l in aln.header_text.splitlines() if not l.startswith("@PG")], open(j(tag + ".tsv"), "rb").read()] + \
            _body(j(tag + ".vcf"), "##source") + [open(j(tag + ".fas")).read().split("\n", 1)]
    a, b_ = outs["plain"], outs["flag"]
    assert a[:-1] == b_[:-1]
    assert a[-1][1] == b_[-1][1] and a[-1][0] == ">sample" and b_[-1][0] == ">" + p


@pytest.mark.gpu
def test_gpu_cli_rejects_unknown_contig_with_reads(tmp_path, segs):
    small = [dict(s, b=s["b"].take(np.arange(500))) for s in segs[:2]]
    b, sid = _combined(small, n_unmapped=0)
    d = str(tmp_path)
    j = _split_inputs(d, small, b, sid, "bam")
    with open(j("one.fas"), "w") as f:                               # seg2 is not in this FASTA
        f.write(">%s\n%s\n" % (small[0]["id"], small[0]["g"]))
    with open(j("one.bed"), "w") as f:
        f.write("%s\t10\t30\tp\n" % small[0]["id"])
    with pytest.raises(SystemExit):
        cli.main(["aio", "--multi_contig", "-i", j("multi.bam"), "-p", j("one.bed"), "-r", j("one.fas"), "-ot", j("o.bam"), "-ov", j("o.vcf"),
                  "-oc", j("o.fas")])
