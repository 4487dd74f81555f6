"""iVar-format outputs (DESIGN.md 3.7): the strand / quality pass and the iVar calling of amp_ivar.cuh, their C ABI and the
command line's --output_tsv / --iupac_threshold.

CPU: the kernels' own source on the emulator (tests/emu/amp_emu_ivar.cpp) against a serial C reference of the pass
(tests/stats_oracle.c) and a Python form of the calling; p-values against exact rational arithmetic and scipy.
GPU: the same through the C ABI on config-2 and ONT-like batches."""
import ctypes
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import emu_driver
import golden_io
import parity
from amplipy_b200 import calling, cli, ivar, synth
from amplipy_b200.calling import CallResult
from amplipy_b200.primers import find_overlapping_primers, max_primer_len

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "amplipy_b200", "csrc")
_p = emu_driver._p


# ---------------------------------------------------------------------------------------------------------------- builds
@pytest.fixture(scope="module")
def builds():
    """The emulator with amp_ivar.cuh and the serial reference of the pass, built into a temporary directory."""
    d = tempfile.mkdtemp(prefix="amp_ivar_test_")
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
    gcc = "/usr/bin/gcc" if os.path.isfile("/usr/bin/gcc") else "gcc"
    emu = os.path.join(d, "libamp_emu_ivar.so")
    subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2", "-o", emu,
                           os.path.join(_HERE, "emu", "amp_emu_ivar.cpp")])
    orc = os.path.join(d, "libstats_oracle.so")
    subprocess.check_call([gcc, "-O2", "-fPIC", "-shared", "-o", orc, os.path.join(_HERE, "stats_oracle.c")])
    lib = ctypes.CDLL(emu)
    lib.emu_create.restype = ctypes.c_void_p
    lib.emu_ins_count.restype = ctypes.c_longlong
    lib.emu_ins_chars.restype = ctypes.c_longlong
    lib.emu_error_flags.restype = ctypes.c_uint
    lib.emu_fisher_less.restype = ctypes.c_double
    lib.emu_fisher_less.argtypes = [ctypes.c_longlong, ctypes.c_longlong, ctypes.c_int]
    olib = ctypes.CDLL(orc)
    olib.oracle_pileup_stats_batch.restype = ctypes.c_int64
    yield lib, olib
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture
def emu(builds, monkeypatch):
    monkeypatch.setattr(emu_driver, "lib", lambda: builds[0])
    return builds[0]


# ---------------------------------------------------------------------------------------------------------------- references
def oracle_stats(olib, b, L, minq, trimmed=None):
    """Serial strand / quality sums: rev, qsum int64[6, L] and {(pos, key): [rev, qsum, head]} of the insertion alleles."""
    rev = np.zeros((6, L), np.int64)
    qsum = np.zeros((6, L), np.int64)
    if trimmed is None:
        pos, cigar, ncig, stride3, skip = b.pos, b.cigar, None, 0, None
    else:
        pos, cigar, ncig, stride3, skip = trimmed["pos"], trimmed["cigar"], np.ascontiguousarray(trimmed["ncig"], np.int32), 1, trimmed["flags"]
    cap, ccap = max(int(b.cig_off[-1]), 16), max(int(b.qual_off[-1]), 64)
    while True:
        ev = [np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int8), np.zeros(cap + 1, np.int64),
              np.zeros(ccap, np.uint8)]
        rev[:] = 0
        qsum[:] = 0
        n = int(olib.oracle_pileup_stats_batch(ctypes.c_int64(b.n), _p(pos), _p(b.flag), _p(b.cig_off), _p(cigar), _p(ncig),
                                               ctypes.c_int(stride3), _p(skip), _p(b.seq_off), _p(b.seq), _p(b.qual_off), _p(b.qual),
                                               ctypes.c_int(L), ctypes.c_int(minq), _p(rev), _p(qsum), ctypes.c_int64(cap), _p(ev[0]),
                                               _p(ev[1]), _p(ev[2]), _p(ev[3]), _p(ev[4]), _p(ev[5]), ctypes.c_int64(ccap)))
        if n <= cap and ev[4][n] <= ccap:
            break
        cap, ccap = 2 * max(n, cap), 2 * max(int(ev[4][min(n, cap)]), ccap)
    raw = ev[5].tobytes()
    ins = {}
    for e in range(n):
        key = (int(ev[0][e]), raw[int(ev[4][e]):int(ev[4][e + 1])].decode("latin-1"))
        v = ins.setdefault(key, [0, 0, 0])
        v[0] += int(ev[1][e])
        v[1] += int(ev[2][e])
        v[2] |= int(ev[3][e])
    return rev, qsum, ins


def fisher_exact_less(D, a, mq):
    """P(X <= e) by exact integer arithmetic (the true value, rounded once)."""
    e = math.floor(D * 10 ** (-mq / 10))
    K, M = e + a, 2 * D
    lo, hi = max(0, K - D), min(K, D)
    if e >= hi:
        return 1.0
    return sum(math.comb(K, x) * math.comb(M - K, D - x) for x in range(lo, e + 1)) / math.comb(M, D)


def fisher_scipy_less(D, a, mq):
    from scipy.stats import fisher_exact
    e = math.floor(D * 10 ** (-mq / 10))
    return float(fisher_exact([[e, D - e], [a, D - a]], alternative="less")[1])


def serial_ivar(res, ins, counts, qs, ref_seq, min_depth, min_freq, t, sample=0):
    """The semantics of DESIGN.md 3.7 written out in Python for one sample: (iupac u8[L], fixed_mq [L, 6], fixed_pval [L, 6],
    {k: (mq, pval)}) with NaN = no row.  P-values are exact (math.comb) for D <= 2000, scipy's otherwise."""
    L = res.L
    sl = slice(sample * L, (sample + 1) * L)
    depth = res.depth[sl].astype(np.int64)
    c = counts.astype(np.int64)
    mq = np.zeros((L, 6), np.int64)
    with np.errstate(divide="ignore", invalid="ignore"):
        mq[:, :5] = np.where(c[:5].T > 0, qs.qsum[:5].T // np.maximum(c[:5].T, 1), 0)
        nb = c[:5].sum(0)
        mq[:, 5] = np.where(nb > 0, qs.qsum[:5].sum(0) // np.maximum(nb, 1), 0)
    pval = np.full((L, 6), np.nan)
    ffreq = res.fixed_freq[sl]
    pf = lambda D, a, m: fisher_exact_less(D, a, m) if D <= 2000 else fisher_scipy_less(D, a, m)
    rows = (depth > 0) & (depth >= min_depth)
    for p in np.flatnonzero(rows).tolist():
        for ch in range(6):
            if c[ch, p] and "ACGTN-"[ch] != ref_seq[p] and ffreq[p, ch] >= min_freq:
                pval[p, ch] = pf(int(depth[p]), int(c[ch, p]), int(mq[p, ch]))
    ins_out = {}
    by_pos = {}
    for k in range(ins.k):
        if ins.sample[k] != sample:
            continue
        p, cnt, s = int(ins.pos[k]), int(ins.count[k]), ins.strs[k]
        m = int(qs.ins_qsum[k]) // cnt if cnt else 0
        pv = float("nan")
        if rows[p] and cnt and len(s) > 0 and not (len(s) == 1 and s == ref_seq[p]) and res.ins_freq[k] >= min_freq:
            pv = pf(int(depth[p]), cnt, m)
        ins_out[k] = (m, pv)
        by_pos.setdefault(p, []).append(k)
    iupac = np.zeros(L, np.uint8)
    top, tc = res.top_id[sl], res.top_count[sl]
    codes = "\0ACMGRSVTWYHKDBN"
    for p in range(L):
        if top[p] < 0 or tc[p] < min_depth or tc[p] / depth[p] < min_freq:
            continue
        al = [(int(res.fixed_rank[sample * L + p, ch]), ch, float(ffreq[p, ch])) for ch in range(6) if c[ch, p]]
        al += [(int(res.ins_rank[k]), 6, float(res.ins_freq[k])) for k in by_pos.get(p, ()) if ins.count[k]]
        al.sort()
        tot, pre = 0.0, []
        for _, sym, f in al:
            tot += f
            pre.append(sym)
            if tot >= t:
                break
        if len(pre) > 1:
            if 4 in pre:
                iupac[p] = ord("N")
            else:
                mask = sum(1 << s for s in set(pre) if s < 4)
                iupac[p] = ord(codes[mask]) if mask else 0
    return iupac, mq, pval, ins_out


def check_ivar(got, want, ins, sample=0, L=None):
    iupac, mq, pval, ins_out = want
    L = len(iupac)
    sl = slice(sample * L, (sample + 1) * L)
    assert np.array_equal(got.iupac[sl], iupac), np.flatnonzero(got.iupac[sl] != iupac)[:10]
    assert np.array_equal(got.fixed_mq[sl].astype(np.int64), mq)
    gp = got.fixed_pval[sl]
    assert np.array_equal(np.isnan(gp), np.isnan(pval))
    ok = ~np.isnan(pval)
    np.testing.assert_allclose(gp[ok], pval[ok], rtol=1e-6, atol=0)
    for k, (m, pv) in ins_out.items():
        assert int(got.ins_mq[k]) == m, k
        assert math.isnan(pv) == math.isnan(got.ins_pval[k]), k
        if not math.isnan(pv):
            assert got.ins_pval[k] == pytest.approx(pv, rel=1e-6, abs=0)


def stats_dict(ins, qs, sample=0):
    return {(int(ins.pos[k]), ins.strs[k]): [int(qs.ins_rev[k]), int(qs.ins_qsum[k]), int(qs.ins_head[k])]
            for k in range(ins.k) if ins.sample[k] == sample}


def oracle_ins_only_table(oins, counts_dict):
    """The oracle's per-event dict restricted to the keys the pileup keeps in its table (1-character ACGTN keys are counted in
    the channels, and their stats are in rev / qsum)."""
    return {k: v for k, v in oins.items() if k in counts_dict}


# ---------------------------------------------------------------------------------------------------------------- emulated engine
class EmuIvarEngine(emu_driver.EmuEngine):
    """emu_driver.EmuEngine plus the Engine surface of the iVar outputs, on the kernels' own source."""

    def enable_qstats(self):
        emu_driver.lib().emu_qstats_enable(self._h)
        self._qstats = True

    def process(self, batch, trim=True, pileup=True, sample=0, first=0, n=None, qstats=False, out=None):
        t = super().process(batch, trim=trim, pileup=pileup, sample=sample, first=first, n=n)
        if qstats:
            assert getattr(self, "_qstats", False) and pileup
            n = batch.n - first if n is None else n
            o = (None,) * 4 if t is None else (t.pos, t.ncig, t.flags, t.cigar)
            emu_driver.lib().emu_qstats_pass(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag),
                                             _p(batch.tlen), _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(batch.seq),
                                             _p(batch.qual_off), _p(batch.qual), 1 if trim else 0, sample, *[_p(a) for a in o])
        return t

    def qstats(self, sample=0):
        k = int(emu_driver.lib().emu_ins_count(self._h))
        q = ivar.QStats(np.empty((6, self.L), np.int32), np.empty((6, self.L), np.int64), np.zeros(max(k, 1), np.int32),
                        np.zeros(max(k, 1), np.int64), np.zeros(max(k, 1), np.uint8))
        emu_driver.lib().emu_qstats_host(self._h, sample, _p(q.rev), _p(q.qsum), _p(q.ins_rev), _p(q.ins_qsum), _p(q.ins_head))
        q.ins_rev, q.ins_qsum, q.ins_head = q.ins_rev[:k], q.ins_qsum[:k], q.ins_head[:k]
        return q

    def call(self, ref_seq, *a, **kw):
        self._ref = ref_seq
        self._res = super().call(ref_seq, *a, **kw)
        return self._res

    def call_ivar(self, min_depth=1, min_freq=0.03, iupac_threshold=0.0):
        r = self._res
        k = max(int(emu_driver.lib().emu_ins_count(self._h)), 1)
        SL = self.n_samples * self.L
        out = ivar.IvarResult(np.empty(SL, np.uint8), np.empty((SL, 6), np.int32), np.empty((SL, 6), np.float64), np.zeros(k, np.int32),
                              np.full(k, np.nan))
        emu_driver.lib().emu_call_ivar(self._h, ctypes.c_char_p(self._ref.encode("latin-1")), _p(r.depth), _p(r.top_id), _p(r.top_count),
                                       _p(r.fixed_freq), _p(r.fixed_rank), _p(r.ins_freq), _p(r.ins_rank), int(min_depth),
                                       ctypes.c_double(min_freq), ctypes.c_double(iupac_threshold), _p(out.iupac), _p(out.fixed_mq),
                                       _p(out.fixed_pval), _p(out.ins_mq), _p(out.ins_pval))
        return out


# ---------------------------------------------------------------------------------------------------------------- CPU tests
def _fuzz_batches():
    L = 29903
    g = synth.random_genome(L, 3)
    primers, amps = synth.make_scheme(L, 98, seed=4)
    prim = [(s, e) for s, e, _ in primers]
    return L, g, prim, {"illumina_indels": synth.illumina_batch(g, amps, 3000, seed=31, p_ins=0.08, p_del=0.08),
                        "ont_like": synth.ont_batch(g, amps, 150, seed=32)}


def _check_stats(eng, olib, b, L, minq, trimmed, sample=0):
    rev, qsum, oins = oracle_stats(olib, b, L, minq, trimmed)
    qs = eng.qstats(sample)
    assert np.array_equal(qs.rev.astype(np.int64), rev)
    assert np.array_equal(qs.qsum, qsum)
    ins = eng.insertions()
    got = stats_dict(ins, qs, sample)
    assert got == oracle_ins_only_table(oins, got)
    assert set(got) == set(oracle_ins_only_table(oins, ins.as_dict(sample)))
    assert (eng.error_flags() & 64) == 0


@pytest.mark.parametrize("trim", [True, False])
@pytest.mark.parametrize("name", golden_io.list_cases())
def test_emulated_stats_pass_matches_oracle(name, trim, emu, builds, oracle_lib):
    b, meta, arr = golden_io.load_case(name)
    kw = parity.engine_kwargs(meta)
    eng = EmuIvarEngine(**kw)
    eng.enable_qstats()
    t = eng.process(b, trim=trim, pileup=True, qstats=True)
    trimmed = None
    if trim:
        trimmed = {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags}
    _check_stats(eng, builds[1], b, kw["ref_len"], kw["min_quality"], trimmed)


@pytest.mark.parametrize("minq", [0, 20, 30])
@pytest.mark.parametrize("kind", ["illumina_indels", "ont_like"])
def test_emulated_stats_pass_fuzz(kind, minq, emu, builds):
    L, g, prim, batches = _fuzz_batches()
    b = batches[kind]
    eng = EmuIvarEngine(ref_len=L, primer_tables=find_overlapping_primers(L, prim, 0), max_primer_len=max_primer_len(prim), min_quality=minq,
                        ins_slots=1 << 18, ins_arena_bytes=1 << 24)
    eng.enable_qstats()
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    assert eng.error_flags() == 0
    _check_stats(eng, builds[1], b, L, minq, {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags})


@pytest.mark.parametrize("t", [0.0, 0.5, 0.9, 1.0])
@pytest.mark.parametrize("name", golden_io.list_cases())
def test_emulated_ivar_body_matches_serial_form(name, t, emu):
    b, meta, arr = golden_io.load_case(name)
    p = meta["params"]
    eng = EmuIvarEngine(**parity.engine_kwargs(meta))
    eng.enable_qstats()
    eng.process(b, trim=True, pileup=True, qstats=True)
    ref = bytes(arr["ref_seq"]).decode()
    res = eng.call(ref, p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"], p["min_freq_variants"])
    md, mf = (p["min_depth_variants"], p["min_freq_variants"]) if t in (0.0, 1.0) else (p["min_depth_consensus"], p["min_freq_consensus"])
    got = eng.call_ivar(md, mf, t)
    check_ivar(got, serial_ivar(res, eng.insertions(), eng.counts(), eng.qstats(), ref, md, mf, t), eng.insertions())


def test_pval_against_exact_and_scipy(builds):
    lib = builds[0]
    rng = np.random.default_rng(5)
    cases = [(1, 1, 0), (10, 10, 0), (10, 1, 0), (5, 3, 40), (2000, 1, 30), (2000, 1999, 2), (1, 1, 93), (7, 2, 255)]
    for _ in range(300):
        D = int(rng.integers(1, 2001))
        cases.append((D, int(rng.integers(1, D + 1)), int(rng.integers(0, 45))))
    for D, a, mq in cases:
        want = fisher_exact_less(D, a, mq)
        got = lib.emu_fisher_less(D, a, mq)
        if want >= 1e-300:
            assert got == pytest.approx(want, rel=1e-6, abs=0), (D, a, mq)
        else:
            assert got < 1e-290, (D, a, mq)
    for _ in range(40):
        D = int(rng.integers(2001, 200000))
        a, mq = int(rng.integers(1, D + 1)), int(rng.integers(0, 45))
        for aa in (a, max(1, int(D * 10 ** (-mq / 10))) + int(rng.integers(0, 3))):
            aa = min(aa, D)
            want = fisher_scipy_less(D, aa, mq)
            if want >= 1e-300:
                assert lib.emu_fisher_less(D, aa, mq) == pytest.approx(want, rel=1e-6, abs=0), (D, aa, mq)


# ---------------------------------------------------------------------------------------------------------------- CLI
GOLD = os.path.join(_HERE, "golden", "cli")


def _aio(tmp, tag, extra):
    j = lambda n: os.path.join(tmp, n)
    for f in ("in.sam", "primers.bed", "ref.fas"):
        if not os.path.isfile(j(f)):
            shutil.copy(os.path.join(GOLD, f), tmp)
    cli.main(["aio", "-i", j("in.sam"), "-p", j("primers.bed"), "-r", j("ref.fas"), "-ot", j(tag + ".sam"), "-ov", j(tag + ".vcf"),
              "-oc", j(tag + ".fas"), "-mfc", "0.2", "-mdc", "3"] + extra)
    return j


def _vcf_body(path):
    return [l for l in open(path) if not l.startswith("##source")]


def test_cli_tsv_and_iupac_match_reference(tmp_path, emu, builds, monkeypatch):
    import amplipy_b200.engine as engine_mod
    monkeypatch.setattr(engine_mod, "Engine", EmuIvarEngine)
    d = str(tmp_path)
    j = _aio(d, "plain", [])
    _aio(d, "ivar", ["--output_tsv", j("ivar.tsv"), "--iupac_threshold", "0.6"])
    _aio(d, "zero", ["--iupac_threshold", "0"])
    assert open(j("zero.fas"), "rb").read() == open(j("plain.fas"), "rb").read()
    assert _vcf_body(j("ivar.vcf")) == _vcf_body(j("plain.vcf"))
    # the Python reference: oracle counts and stats of the trimmed reads, the calling of the emulated engine
    from amplipy_b200 import alnio
    ref_id, ref = cli.load_ref_genome(j("ref.fas"))
    L = len(ref)
    aln = alnio.read_alignments(j("in.sam"))
    from amplipy_b200.primers import load_primers
    prim = load_primers(j("primers.bed"))
    eng = EmuIvarEngine(ref_len=L, primer_tables=find_overlapping_primers(L, prim, 0), max_primer_len=max_primer_len(prim))
    eng.enable_qstats()
    t = eng.process(aln.batch, trim=True, pileup=True, qstats=True)
    counts = eng.counts()
    ins = eng.insertions()
    rev, qsum, oins = oracle_stats(builds[1], aln.batch, L, 20, {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags})
    qs = ivar.QStats(rev.astype(np.int32), qsum, np.array([oins[(int(ins.pos[k]), ins.strs[k])][0] for k in range(ins.k)], np.int32),
                     np.array([oins[(int(ins.pos[k]), ins.strs[k])][1] for k in range(ins.k)], np.int64),
                     np.array([oins[(int(ins.pos[k]), ins.strs[k])][2] for k in range(ins.k)], np.uint8))
    res = eng.call(ref, 3, 0.2, 1, 0.03)
    want_v = serial_ivar(res, ins, counts, qs, ref, 1, 0.03, 0.0)
    iv = ivar.IvarResult(want_v[0], want_v[1].astype(np.int32), want_v[2], np.zeros(max(ins.k, 1), np.int32), np.full(max(ins.k, 1), np.nan))
    for k, (m, pv) in want_v[3].items():
        iv.ins_mq[k], iv.ins_pval[k] = m, pv
    rows = ivar.tsv_rows(res, ins, iv, qs, ref_id, ref, counts)
    assert len(rows) > 0
    got = open(j("ivar.tsv")).read().splitlines()
    assert got[0].split("\t") == list(ivar.TSV_HEADER)
    assert len(got) - 1 == len(rows)
    for line, r in zip(got[1:], rows):
        f = line.split("\t")
        want = ivar.format_row(r).split("\t")
        assert f[:12] == want[:12] and f[13:] == want[13:], (f, want)
        assert float(f[12]) == pytest.approx(float(want[12]), rel=1e-6)
    want_c = serial_ivar(res, ins, counts, qs, ref, 3, 0.2, 0.6)[0]
    want_fas = ">sample\n%s\n" % calling.consensus_string(res, ins, 0, "N", iupac=want_c)
    assert open(j("ivar.fas")).read() == want_fas


def test_cli_rejects_bad_threshold_and_existing_tsv(tmp_path, emu, monkeypatch):
    import amplipy_b200.engine as engine_mod
    monkeypatch.setattr(engine_mod, "Engine", EmuIvarEngine)
    d = str(tmp_path)
    with pytest.raises(SystemExit):
        _aio(d, "a", ["--iupac_threshold", "1.5"])
    open(os.path.join(d, "x.tsv"), "w").close()
    with pytest.raises(SystemExit):
        _aio(d, "b", ["--output_tsv", os.path.join(d, "x.tsv")])


def test_alt_text():
    assert ivar.alt_text("G", "A") == "G"
    assert ivar.alt_text("-", "A") == "-A"
    assert ivar.alt_text("ACGT", "A") == "+CGT"
    assert ivar.alt_text("CGTA", "A", head=True) == "+CGT"


# ---------------------------------------------------------------------------------------------------------------- GPU
GL = 29903


@pytest.fixture(scope="module")
def gpu_workload():
    g = synth.random_genome(GL, 7)
    primers, amps = synth.make_scheme(GL, 98, seed=2)
    prim = [(s, e) for s, e, _ in primers]
    snvs = [(1000 + 2800 * i, "ACGT"[i % 4], af) for i, af in enumerate([1.0, 0.9, 0.75, 0.5, 0.4, 0.3, 0.2, 0.1, 0.05, 0.05])]
    return dict(g=g, amps=amps, prim=prim, tables=find_overlapping_primers(GL, prim, 0), mpl=max_primer_len(prim),
                cfg2=synth.illumina_batch(g, amps, 1_000_000, seed=1, snvs=snvs), ont=synth.ont_batch(g, amps, 40_000, seed=4))


def _gpu_engine(w, n_samples=1, big=False):
    from amplipy_b200.engine import Engine
    return Engine(ref_len=GL, primer_tables=w["tables"], max_primer_len=w["mpl"], device=0, n_samples=n_samples,
                  ins_slots=(1 << 24) if big else 0, ins_arena_bytes=(1 << 30) if big else 0)


def _trim_dict(t):
    return {"pos": t.pos, "ncig": t.ncig, "cigar": t.cigar, "flags": t.flags}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["cfg2", "ont"])
def test_gpu_stats_strand_split_and_oracle(kind, gpu_workload, builds):
    w = gpu_workload
    b = w[kind]
    big = kind == "ont"
    eng = _gpu_engine(w, big=big)
    eng.enable_qstats()
    t = eng.process(b, trim=True, pileup=True, qstats=True)
    assert eng.error_flags() == 0
    qs, ins = eng.qstats(), eng.insertions()
    # rev = the count matrix of a run over the reverse-strand reads alone; ins_rev = that run's insertion counts
    r = _gpu_engine(w, big=big)
    r.process(b.take(np.flatnonzero(b.flag & 16)), trim=True, pileup=True)
    assert np.array_equal(qs.rev, r.counts())
    rins = r.insertions().as_dict()
    got = {(int(ins.pos[k]), ins.strs[k]): int(qs.ins_rev[k]) for k in range(ins.k)}
    assert {k: v for k, v in got.items() if v} == rins
    rev, qsum, oins = oracle_stats(builds[1], b, GL, 20, _trim_dict(t))
    assert np.array_equal(qs.qsum, qsum) and np.array_equal(qs.rev.astype(np.int64), rev)
    assert stats_dict(ins, qs) == oracle_ins_only_table(oins, ins.as_dict())


@pytest.mark.gpu
def test_gpu_qstats_leaves_every_other_output_unchanged(gpu_workload):
    w = gpu_workload
    for kind in ("cfg2", "ont"):
        b = w[kind]
        outs = []
        for qstats in (False, True):
            eng = _gpu_engine(w, big=kind == "ont")
            if qstats:
                eng.enable_qstats()
            t = eng.process(b, trim=True, pileup=True, qstats=qstats)
            res = eng.call(w["g"])
            ins = eng.insertions()
            outs.append([t.pos.tobytes(), t.ncig.tobytes(), t.flags.tobytes(), t.cigar.tobytes(), eng.counts().tobytes(),
                         sorted(ins.as_dict().items())] + [np.ascontiguousarray(getattr(res, f)).tobytes() for f in
                                                            ("depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask")])
            assert eng.error_flags() == 0
            eng.close()
        assert outs[0] == outs[1], kind


@pytest.mark.gpu
def test_gpu_host_device_decoded_paths_agree(gpu_workload):
    from amplipy_b200 import alnio
    w = gpu_workload
    b = w["cfg2"].take(np.arange(200_000))
    eng = _gpu_engine(w)
    eng.enable_qstats()
    eng.process(b, trim=True, pileup=True, qstats=True)
    ref = eng.qstats(), eng.insertions()
    want = (ref[0].rev.tobytes(), ref[0].qsum.tobytes(), stats_dict(ref[1], ref[0]))
    eng.reset()
    d = eng.upload(b)
    eng.process_device(d, trim=True, pileup=True, qstats=True)
    q, i = eng.qstats(), eng.insertions()
    assert (q.rev.tobytes(), q.qsum.tobytes(), stats_dict(i, q)) == want
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "x.bam")
        alnio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ref\tLN:%d\n" % GL, [("ref", GL)], b)
        raw = open(path, "rb").read()
    eng.reset_async()
    eng.decode_bam(raw, alnio.bam_layout(raw))
    eng.process_decoded(trim=True, pileup=True, qstats=True)
    q, i = eng.qstats(), eng.insertions()
    assert (q.rev.tobytes(), q.qsum.tobytes(), stats_dict(i, q)) == want
    assert eng.error_flags() == 0


@pytest.mark.gpu
def test_gpu_plate_equals_solo_runs_and_ivar_calling(gpu_workload, builds):
    w = gpu_workload
    parts = [w["cfg2"].take(np.arange(k * 100_000, (k + 1) * 100_000)) for k in range(2)] + [w["ont"].take(np.arange(5_000))]
    plate = _gpu_engine(w, n_samples=3, big=True)
    plate.enable_qstats()
    for s, b in enumerate(parts):
        plate.process(b, trim=True, pileup=True, sample=s, qstats=True)
    res = plate.call(w["g"])
    pins = plate.insertions()
    iv = plate.call_ivar(1, 0.03, 0.0)
    ivc = plate.call_ivar(10, 0.0, 0.7)
    assert plate.error_flags() == 0
    for s, b in enumerate(parts):
        solo = _gpu_engine(w, big=True)
        solo.enable_qstats()
        solo.process(b, trim=True, pileup=True, qstats=True)
        q, sq = solo.qstats(), plate.qstats(s)
        assert np.array_equal(q.rev, sq.rev) and np.array_equal(q.qsum, sq.qsum)
        assert stats_dict(solo.insertions(), q) == stats_dict(pins, sq, s)
        sres = solo.call(w["g"])
        sins = solo.insertions()
        for (mdp, mf, t), piv in (((1, 0.03, 0.0), iv), ((10, 0.0, 0.7), ivc)):
            siv = solo.call_ivar(mdp, mf, t)
            check_ivar(siv, serial_ivar(sres, sins, solo.counts(), q, w["g"], mdp, mf, t), sins)
            sl = slice(s * GL, (s + 1) * GL)
            assert np.array_equal(piv.iupac[sl], siv.iupac) and np.array_equal(piv.fixed_mq[sl], siv.fixed_mq)
            assert piv.fixed_pval[sl].tobytes() == siv.fixed_pval.tobytes()
        solo.close()


@pytest.mark.gpu
def test_gpu_state_errors(gpu_workload):
    from amplipy_b200.engine import AmpError
    w = gpu_workload
    eng = _gpu_engine(w)
    b = w["cfg2"].take(np.arange(1000))
    with pytest.raises(AmpError):
        eng.process(b, trim=True, pileup=True, qstats=True)          # not enabled
    eng.enable_qstats()
    with pytest.raises(AmpError):
        eng.process(b, trim=True, pileup=False, qstats=True)         # no pileup
    with pytest.raises(AmpError):
        eng.allreduce_counts(1)
    eng.process(b, trim=True, pileup=True, qstats=True)
    eng.call(w["g"])
    with pytest.raises(AmpError):
        eng.call_ivar(1, 0.03, 1.5)
