"""Codon annotation of the iVar TSV (DESIGN.md 3.9): the GFF3 loader, the annotation of amp_annot.cuh, its C ABI and the command
line's --gff.

CPU: the loader and its errors; the kernels' own source on the emulator (tests/emu/amp_emu_annot.cpp) against a Python form of
the rules written out below; known answers; the CLI on the emulated engine.
GPU: the same through the C ABI, a plate against solo runs, --multi_contig against single-contig runs, the ABI's error codes."""
import ctypes
import gzip
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import emu_driver
from amplipy_b200 import cli, gff, ivar, synth
from amplipy_b200.gff import Feature
from amplipy_b200.primers import InputError
from test_contig import _body, _combined, _split_inputs, segs  # noqa: F401  (segs: the contigs fixture)
from test_ivar import EmuIvarEngine, _aio

_HERE = os.path.dirname(os.path.abspath(__file__))
_p = emu_driver._p
CODE1 = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"


# ---------------------------------------------------------------------------------------------------------------- Python form
def translate(c):
    if any(b not in "TCAG" for b in c):
        return "X"
    return CODE1[16 * "TCAG".index(c[0]) + 4 * "TCAG".index(c[1]) + "TCAG".index(c[2])]


def comp(b):
    return {"A": "T", "T": "A", "C": "G", "G": "C"}.get(b, "N")


def py_annotate(refs, features, L):
    """The rules of DESIGN.md 3.9 for samples with references refs[s] and features features[s]: {gp: [(feature index, POS_AA,
    offset, 18 codon characters, 6 amino acids)]} in occurrence order."""
    occ = {}
    for s, (ref, feats) in enumerate(zip(refs, features)):
        for fi, ft in enumerate(feats):
            segs_ = sorted(ft.segments, key=lambda x: x[0] * ft.strand)            # 5' to 3'
            coords = []
            for lo, hi in segs_:
                coords += list(range(lo, hi)) if ft.strand > 0 else list(range(hi - 1, lo - 1, -1))
            cds = coords[ft.phase:]
            for i in range(len(cds) // 3):
                gs = cds[3 * i:3 * i + 3]
                cod = "".join(ref[g].upper() if ft.strand > 0 else comp(ref[g].upper()) for g in gs)
                for k, g in enumerate(gs):
                    codons, aas = cod, translate(cod)
                    for x in "ACGTN":
                        b = x if ft.strand > 0 else comp(x)
                        alt = cod[:k] + b + cod[k + 1:]
                        codons += alt
                        aas += translate(alt)
                    occ.setdefault(s * L + g, []).append((fi, i + 1, k, codons, aas))
    return occ


def ann_as_dict(a):
    out = {}
    for gp in np.flatnonzero(np.diff(a.off.astype(np.int64))).tolist():
        out[gp] = [(int(a.feat[e]), int(a.pos_aa[e]), int(a.codon_off[e]), a.codons[e].tobytes().decode(), a.aas[e].tobytes().decode())
                   for e in range(int(a.off[gp]), int(a.off[gp + 1]))]
    return out


# ---------------------------------------------------------------------------------------------------------------- emulator
@pytest.fixture(scope="module")
def alib():
    d = tempfile.mkdtemp(prefix="amp_annot_test_")
    gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
    so = os.path.join(d, "libamp_emu_annot.so")
    subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2", "-o", so,
                           os.path.join(_HERE, "emu", "amp_emu_annot.cpp")])
    lib = ctypes.CDLL(so)
    for n, t in (("emu_create", ctypes.c_void_p), ("emu_ins_count", ctypes.c_longlong), ("emu_ins_chars", ctypes.c_longlong),
                 ("emu_error_flags", ctypes.c_uint), ("emu_annot_build", ctypes.c_longlong)):
        getattr(lib, n).restype = t
    yield lib
    shutil.rmtree(d, ignore_errors=True)


def emu_annotate(lib, refs, features, L, shared_ref=False):
    """amp_annotate on the emulator: refs[s] padded with 'N' to L (or one reference for all samples, ``shared_ref``)."""
    S = len(features)
    buf = (refs[0] if shared_ref else "".join(r + "N" * (L - len(r)) for r in refs)).encode("latin-1")
    lens = np.array([len(refs[0] if shared_ref else r) for r in refs] if not shared_ref else [len(refs[0])] * S, np.int32)
    flat = [f for fs in features for f in fs]
    nf = np.array([len(fs) for fs in features], np.int32)
    strand = np.array([f.strand for f in flat] + [0], np.int32)
    phase = np.array([f.phase for f in flat] + [0], np.int32)
    seg_off = np.zeros(len(flat) + 1, np.int32)
    np.cumsum([len(f.segments) for f in flat], out=seg_off[1:])
    start = np.array([s for f in flat for s, _ in f.segments] + [0], np.int32)
    end = np.array([e for f in flat for _, e in f.segments] + [0], np.int32)
    E = int(lib.emu_annot_build(S, L, ctypes.c_char_p(buf), ctypes.c_longlong(0 if shared_ref else L), _p(lens), _p(nf), _p(strand),
                                _p(phase), _p(seg_off), _p(start), _p(end)))
    if E < 0:
        return None
    k = max(E, 1)
    a = ivar.Annotation(L, np.empty(S * L + 1, np.uint32), np.empty(k, np.int32), np.empty(k, np.int32), np.empty(k, np.uint8),
                        np.empty((k, 18), np.uint8), np.empty((k, 6), np.uint8))
    lib.emu_annot_copy(_p(a.off), _p(a.feat), _p(a.pos_aa), _p(a.codon_off), _p(a.codons), _p(a.aas))
    a.feat, a.pos_aa, a.codon_off, a.codons, a.aas = a.feat[:E], a.pos_aa[:E], a.codon_off[:E], a.codons[:E], a.aas[:E]
    return a


def random_ref(L, seed):
    rng = np.random.default_rng(seed)
    s = np.array(list("ACGT"), dtype="<U1")[rng.integers(0, 4, L)]
    s[rng.random(L) < 0.1] = "N"
    low = rng.random(L) < 0.2
    s[low] = np.char.lower(s[low])
    s[rng.random(L) < 0.01] = "R"                   # an IUPAC code in the FASTA
    return "".join(s.tolist())


def hand_features(L):
    """'+' and '-', phases 0 / 1 / 2, the ORF1ab shape (1-base overlap), overlapping features, a trailing partial codon and
    features at the first and last base of a contig of length L."""
    F = lambda n, st, ph, sg: Feature(n, "c", st, ph, sorted(sg, key=lambda x: x[0] * st))
    return [F("orf1ab", 1, 0, [(10, 61), (60, 130)]), F("first", 1, 0, [(0, 12)]), F("rev", -1, 0, [(40, 100)]),
            F("rev_spliced", -1, 2, [(150, 170), (120, 140)]), F("ph1", 1, 1, [(200, 231)]), F("ph2", -1, 2, [(205, 241)]),
            F("partial", 1, 0, [(250, 264)]), F("nested", 1, 0, [(215, 227)]), F("last", -1, 1, [(L - 20, L)]),
            F("last_fwd", 1, 0, [(L - 9, L)])]


# ---------------------------------------------------------------------------------------------------------------- CPU: loader
def _write(path, text):
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "wt") as f:
        f.write(text)
    return path


GFF_TEXT = ("##gff-version 3\n#comment\nref\tsrc\tgene\t1\t100\t.\t+\t.\tID=gene-1\n"
            "ref\tsrc\tCDS\t10\t30\t.\t+\t0\tID=cds-ORF1ab;Parent=gene-1\n"
            "ref\tsrc\tCDS\t60\t90\t.\t-\t.\tParent=S%3Bspike%2C2;Name=x\n"
            "ref\tsrc\tCDS\t30\t45\t.\t+\t2\tID=cds-ORF1ab\n"
            "ref\tsrc\tCDS\t100\t120\t.\t-\t1\tParent=S%3Bspike%2C2\n"
            "\n##FASTA\n>ref\nACGT\nnot a gff line\n")


@pytest.mark.parametrize("gz", [False, True])
def test_load_gff_grouping_decoding_and_fasta(tmp_path, gz):
    fts = gff.load_gff(_write(str(tmp_path / ("a.gff" + (".gz" if gz else ""))), GFF_TEXT))
    assert [f.name for f in fts] == ["cds-ORF1ab", "S;spike,2"]
    a, b = fts
    assert (a.strand, a.phase, a.segments) == (1, 0, [(9, 30), (29, 45)])
    assert (b.strand, b.phase, b.segments) == (-1, 1, [(99, 120), (59, 90)])   # 5' to 3' on '-': the phase of the 100..120 row
    assert a.seqid == b.seqid == "ref"


@pytest.mark.parametrize("line,msg", [
    ("ref\tsrc\tCDS\t10\t30\t.\t+\t0", gff.ERROR_TEXT_INVALID_GFF_LINE),
    ("ref\tsrc\tCDS\tx\t30\t.\t+\t0\tID=a", gff.ERROR_TEXT_INVALID_GFF_COORDS),
    ("ref\tsrc\tCDS\t0\t30\t.\t+\t0\tID=a", gff.ERROR_TEXT_INVALID_GFF_COORDS),
    ("ref\tsrc\tCDS\t31\t30\t.\t+\t0\tID=a", gff.ERROR_TEXT_INVALID_GFF_COORDS),
    ("ref\tsrc\tCDS\t10\t30\t.\t.\t0\tID=a", gff.ERROR_TEXT_INVALID_GFF_STRAND),
    ("ref\tsrc\tCDS\t10\t30\t.\t+\t3\tID=a", gff.ERROR_TEXT_INVALID_GFF_PHASE),
    ("ref\tsrc\tCDS\t10\t30\t.\t+\t0\tName=a", gff.ERROR_TEXT_GFF_NO_ID),
    ("ref\tsrc\tCDS\t10\t30\t.\t+\t0\tID=a\nref\tsrc\tCDS\t40\t50\t.\t-\t0\tID=a", gff.ERROR_TEXT_GFF_MIXED),
    ("ref\tsrc\tCDS\t10\t30\t.\t+\t0\tID=a\nchr2\tsrc\tCDS\t40\t50\t.\t+\t0\tID=a", gff.ERROR_TEXT_GFF_MIXED),
    ("ref\tsrc\tgene\t10\t30\t.\t+\t.\tID=a", gff.ERROR_TEXT_GFF_NO_CDS),
])
def test_load_gff_errors(tmp_path, line, msg):
    with pytest.raises(InputError, match=msg.replace("(", r"\(")):
        gff.load_gff(_write(str(tmp_path / "b.gff"), "##gff-version 3\n" + line + "\n"))


def test_load_gff_missing_file(tmp_path):
    with pytest.raises(InputError, match=gff.ERROR_TEXT_FILE_NOT_FOUND):
        gff.load_gff(str(tmp_path / "nope.gff"))


def test_seqid_rules():
    a, b = Feature("a", "c1", 1, 0, [(0, 9)]), Feature("b", "c2", -1, 0, [(3, 30)])
    contigs = [("c1", "A" * 20), ("c2", "C" * 40)]
    assert gff.features_by_contig([a, b], contigs, True) == [[a], [b]]
    with pytest.raises(InputError, match=gff.ERROR_TEXT_GFF_SEQID_NOT_IN_FASTA):
        gff.features_by_contig([Feature("x", "c9", 1, 0, [(0, 3)])], contigs, True)
    with pytest.raises(InputError, match=gff.ERROR_TEXT_GFF_PAST_END):
        gff.features_by_contig([Feature("x", "c1", 1, 0, [(0, 21)])], contigs, True)
    # without --multi_contig the seqid is ignored, but the rows must name one sequence
    assert gff.features_by_contig([Feature("x", "other", 1, 0, [(0, 3)])], [("c1", "A" * 20)], False)[0][0].name == "x"
    with pytest.raises(InputError, match="use --multi_contig"):
        gff.features_by_contig([a, b], [("c1", "A" * 40)], False)
    with pytest.raises(InputError, match=gff.ERROR_TEXT_GFF_PAST_END):
        gff.features_by_contig([b], [("c1", "A" * 29)], False)


# ---------------------------------------------------------------------------------------------------------------- CPU: emulator
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_emulated_annotation_matches_python_form(alib, seed):
    L = 400
    lens = [400, 333, 287]                                      # contigs shorter than the context
    refs = [random_ref(n, 10 * seed + k) for k, n in enumerate(lens)]
    feats = [hand_features(n) for n in lens]
    feats[2] = feats[2][::-1][:6]                               # another order, fewer features
    rng = np.random.default_rng(seed)
    for k, n in enumerate(lens):                                # and random ones
        for r in range(12):
            st = 1 if rng.random() < 0.5 else -1
            nseg = int(rng.integers(1, 4))
            sg = []
            for _ in range(nseg):
                lo = int(rng.integers(0, n - 1))
                sg.append((lo, int(rng.integers(lo + 1, min(n, lo + 90) + 1))))
            feats[k].append(Feature("r%d" % r, "c", st, int(rng.integers(0, 3)), sorted(sg, key=lambda x: x[0] * st)))
    got = emu_annotate(alib, refs, feats, L)
    want = py_annotate(refs, feats, L)
    assert ann_as_dict(got) == want
    assert len(got.feat) == sum(len(v) for v in want.values()) > 0


def test_emulated_shared_reference_and_empty_samples(alib):
    ref = random_ref(300, 7)
    feats = [hand_features(300), [], hand_features(300)[3:]]
    got = emu_annotate(alib, [ref] * 3, feats, 300, shared_ref=True)
    assert ann_as_dict(got) == py_annotate([ref] * 3, feats, 300)
    assert int(got.off[600]) == int(got.off[300])               # sample 1 has no occurrences


def test_known_answers(alib):
    ref = "ATGGATTAA"
    a = ann_as_dict(emu_annotate(alib, [ref], [[Feature("f", "c", 1, 0, [(0, 9)])]], 9))
    fi, pos_aa, k, cod, aa = a[4][0]
    assert (pos_aa, k, cod[:3], aa[0]) == (2, 1, "GAT", "D")
    assert (cod[3 + 3:6 + 3], aa[1 + 1]) == ("GCT", "A")        # C at the D codon's second base: D2A
    assert aa == "D" + "".join(translate("G" + x + "T") for x in "ACGTN") == "DDAGVX"
    assert a[0][0][4][0] == "M" and a[8][0][4][0] == "*"
    # the same gene on the reverse strand: reverse complement of ref, feature on '-'
    rc = "".join(comp(b) for b in ref[::-1])                    # TTAATCCAT
    b = ann_as_dict(emu_annotate(alib, [rc], [[Feature("f", "c", -1, 0, [(0, 9)])]], 9))
    fi, pos_aa, k, cod, aa = b[4][0]
    assert (pos_aa, k, cod[:3], aa[0]) == (2, 1, "GAT", "D")
    assert (cod[3 + 3 * "ACGTN".index("G"):6 + 3 * "ACGTN".index("G")], aa[1 + "ACGTN".index("G")]) == ("GCT", "A")   # G on '+' = C
    assert b[8][0][4][0] == "M" and b[0][0][4][0] == "*"


def test_emulated_rejects_bad_features(alib):
    ref = "ACGT" * 10
    bad = [Feature("a", "c", 1, 3, [(0, 9)]), Feature("a", "c", 2, 0, [(0, 9)]), Feature("a", "c", 1, 0, [(5, 5)]),
           Feature("a", "c", 1, 0, [(-1, 5)]), Feature("a", "c", 1, 0, [(0, 41)]), Feature("a", "c", 1, 0, [])]
    for f in bad:
        assert emu_annotate(alib, [ref], [[f]], 40) is None, f
    assert emu_annotate(alib, [ref], [[Feature("a", "c", 1, 0, [(0, 40)])]], 40) is not None


# ---------------------------------------------------------------------------------------------------------------- CPU: CLI
class EmuAnnotEngine(EmuIvarEngine):
    """EmuIvarEngine plus set_features / annotate on amp_annot.cuh's source."""

    def set_features(self, sample, features):
        assert getattr(self, "_ref", None) is not None           # the reference comes with call(), as on the device
        self._feats = getattr(self, "_feats", {})
        self._feats[sample] = list(features)

    def annotate(self):
        feats = [self._feats.get(s, []) for s in range(self.n_samples)]
        return emu_annotate(emu_driver.lib(), [self._ref] * self.n_samples, feats, self.L, shared_ref=True)


def _gff_for_cli(path):
    """CDS features on the 4000-base CLI reference: '+' and '-', a phase, the ORF1ab shape, overlaps."""
    rows = [("CDS", 30, 1400, "+", "0", "ID=orf1;Name=ORF1"), ("CDS", 1400, 2200, "+", "0", "ID=orf1"),
            ("CDS", 500, 1100, "-", "1", "Parent=rna-N"), ("CDS", 2300, 3999, "+", "2", "ID=S%20gene"),
            ("CDS", 2600, 2900, "-", "0", "ID=nested")]
    with open(path, "w") as f:
        f.write("##gff-version 3\n" + "".join("synth_ref\tt\t%s\t%d\t%d\t.\t%s\t%s\t%s\n" % r for r in rows))
    return path


def _split_tsv(path):
    return [l.split("\t") for l in open(path).read().splitlines()[1:]]


def test_cli_gff_matches_python_form(tmp_path, alib, monkeypatch):
    import amplipy_b200.engine as engine_mod
    monkeypatch.setattr(emu_driver, "lib", lambda: alib)
    monkeypatch.setattr(engine_mod, "Engine", EmuAnnotEngine)
    d = str(tmp_path)
    g = _gff_for_cli(os.path.join(d, "a.gff"))
    j = _aio(d, "plain", ["--output_tsv", os.path.join(d, "plain.tsv")])
    _aio(d, "ann", ["--output_tsv", j("ann.tsv"), "--gff", g])
    for ext in (".vcf", ".fas", ".sam"):
        a, b = open(j("plain" + ext)).read(), open(j("ann" + ext)).read()
        if ext == ".sam":                                          # the @PG line carries the command line
            a, b = [[l for l in x.splitlines() if not l.startswith("@PG")] for x in (a, b)]
        elif ext == ".vcf":
            a, b = [[l for l in x.splitlines() if not l.startswith("##source")] for x in (a, b)]
        assert a == b, ext
    ref_id, ref = cli.load_ref_genome(j("ref.fas"))
    feats = gff.features_by_contig(gff.load_gff(g), [(ref_id, ref)], False)[0]
    occ = py_annotate([ref], [feats], len(ref))
    plain, got = _split_tsv(j("plain.tsv")), _split_tsv(j("ann.tsv"))
    want = []
    for r in plain:
        o = occ.get(int(r[1]) - 1, [])
        k = "ACGTN".find(r[3]) if len(r[3]) == 1 else -1
        for fi, pos_aa, _, cod, aa in o:
            want.append(r[:14] + [feats[fi].name, cod[:3], aa[0], cod[3 + 3 * k:6 + 3 * k] if k >= 0 else "NA",
                                  aa[1 + k] if k >= 0 else "NA", str(pos_aa)])
        if not o:
            want.append(r)
    assert got == want
    assert len(got) > len(plain) and any(r[14] == "S gene" for r in got) and any(r[3][0] in "+-" and r[14] != "NA" for r in got)
    # dropping the six columns and the repeated rows gives the TSV written without --gff
    dedup = []
    for r in got:
        if not dedup or r[:14] != dedup[-1][:14] or r[14] == "NA":
            dedup.append(r[:14])
    assert dedup == [r[:14] for r in plain] and all(r[14:] == ["NA"] * 6 for r in plain)


def test_cli_gff_needs_tsv(tmp_path, alib, monkeypatch):
    import amplipy_b200.engine as engine_mod
    monkeypatch.setattr(emu_driver, "lib", lambda: alib)
    monkeypatch.setattr(engine_mod, "Engine", EmuAnnotEngine)
    d = str(tmp_path)
    g = _gff_for_cli(os.path.join(d, "a.gff"))
    with pytest.raises(SystemExit):
        _aio(d, "x", ["--gff", g])
    assert not os.path.exists(os.path.join(d, "x.vcf"))
    with pytest.raises(SystemExit):                               # a GFF error is an input error
        _aio(d, "y", ["--output_tsv", os.path.join(d, "y.tsv"), "--gff", os.path.join(d, "missing.gff")])


# ---------------------------------------------------------------------------------------------------------------- GPU
GL = 29903


def _cov2_like_features():
    """A SARS-CoV-2-like layout on a 29,903-base reference: ORF1ab with its -1 frameshift, nested and overlapping ORFs, a
    '-' feature, a phase, a spliced '-' feature."""
    F = lambda n, st, ph, sg: Feature(n, "MN908947.3", st, ph, sorted(sg, key=lambda x: x[0] * st))
    return [F("ORF1ab", 1, 0, [(265, 13468), (13467, 21555)]), F("ORF1a", 1, 0, [(265, 13483)]), F("S", 1, 0, [(21562, 25384)]),
            F("ORF3a", 1, 0, [(25392, 26220)]), F("E", 1, 0, [(26244, 26472)]), F("M", 1, 0, [(26522, 27191)]),
            F("ORF7a", 1, 0, [(27393, 27759)]), F("ORF7b", 1, 0, [(27755, 27887)]), F("N", 1, 0, [(28273, 29533)]),
            F("ORF9b", 1, 0, [(28283, 28577)]), F("antisense", -1, 1, [(20000, 20500), (19000, 19301)]),
            F("ORF10", 1, 2, [(29557, 29674)]), F("tail", -1, 0, [(29890, 29903)])]


@pytest.fixture(scope="module")
def gpu_genome():
    return synth.random_genome(GL, 7)


@pytest.mark.gpu
def test_gpu_annotation_matches_python_form(gpu_genome, alib):
    from amplipy_b200.engine import Engine
    ref = gpu_genome[:5000].lower() + gpu_genome[5000:20000] + "N" * 10 + gpu_genome[20010:]
    feats = _cov2_like_features()
    e = Engine(ref_len=GL)
    e.set_reference(ref)
    e.set_features(0, feats)
    got = e.annotate()
    assert ann_as_dict(got) == py_annotate([ref], [feats], GL)
    emu = emu_annotate(alib, [ref], [feats], GL)
    for f in ("off", "feat", "pos_aa", "codon_off", "codons", "aas"):
        assert np.array_equal(getattr(got, f), getattr(emu, f)), f
    e.close()


@pytest.mark.gpu
def test_gpu_plate_equals_solo_runs(gpu_genome):
    from amplipy_b200.engine import Engine
    S = 24
    rng = np.random.default_rng(3)
    base = _cov2_like_features()
    refs, feats = [], []
    for s in range(S):
        n = GL - int(rng.integers(0, 400))
        g = np.array(list(gpu_genome[:n]))
        mut = rng.random(n) < 0.02
        g[mut] = rng.choice(list("ACGTNacgt"), int(mut.sum()))
        refs.append("".join(g.tolist()))
        fs = [f for f in base if max(e for _, e in f.segments) <= n and rng.random() < 0.8]
        feats.append(fs)
    plate = Engine(ref_len=GL, n_samples=S)
    for s in range(S):
        plate.set_sample_reference(s, refs[s])
        plate.set_features(s, feats[s])
    pa = ann_as_dict(plate.annotate())
    for s in range(S):
        solo = Engine(ref_len=len(refs[s]))
        solo.set_reference(refs[s])
        solo.set_features(0, feats[s])
        sa = ann_as_dict(solo.annotate())
        L = len(refs[s])
        assert {gp - s * GL: v for gp, v in pa.items() if s * GL <= gp < (s + 1) * GL} == {gp % L: v for gp, v in sa.items()}, s
        assert sa == py_annotate([refs[s]], [feats[s]], L)
        solo.close()
    plate.close()


@pytest.mark.gpu
def test_gpu_cli_multi_contig_gff_equals_per_contig_runs(tmp_path, segs):  # noqa: F811
    small = [dict(s, b=s["b"].take(np.arange(min(s["b"].n, 3000)))) for s in segs]
    b, sid = _combined(small, n_unmapped=11)
    d = str(tmp_path)
    j = _split_inputs(d, small, b, sid, "bam")
    rows = []
    for k, s in enumerate(small):
        L = s["L"]
        rows.append((s["id"], "CDS", 20 + k, L - 300, "+", str(k % 3), "ID=%s_p" % s["id"]))
        rows.append((s["id"], "CDS", 100, 400 + k, "-", "0", "Parent=%s_m" % s["id"]))
        rows.append((s["id"], "CDS", 390 + k, L, "-", "1", "Parent=%s_m" % s["id"]))
    body = "".join("%s\tt\t%s\t%d\t%d\t.\t%s\t%s\t%s\n" % r for r in rows)
    with open(j("multi.gff"), "w") as f:
        f.write("##gff-version 3\n" + body)
    for s in small:
        with open(j(s["id"] + ".gff"), "w") as f:
            f.write("##gff-version 3\n" + "".join(l + "\n" for l in body.splitlines() if l.startswith(s["id"] + "\t")))
    cli.main(["aio", "--multi_contig", "-i", j("multi.bam"), "-p", j("multi.bed"), "-r", j("multi.fas"), "-ot", j("m_trim.bam"),
              "-ov", j("m.vcf"), "-oc", j("m.fas"), "--output_tsv", j("m.tsv"), "--gff", j("multi.gff"), "-mdc", "3"])
    want = []
    for s in small:
        p = s["id"]
        cli.main(["aio", "-i", j(p + ".bam"), "-p", j(p + ".bed"), "-r", j(p + ".fas"), "-ot", j(p + "_trim.bam"), "-ov", j(p + ".vcf"),
                  "-oc", j(p + "_c.fas"), "--output_tsv", j(p + ".tsv"), "--gff", j(p + ".gff"), "-mdc", "3"])
        want += _body(j(p + ".tsv"), "REGION")
    got = _body(j("m.tsv"), "REGION")
    assert got == want and len(got) > 0
    assert sum(1 for l in got if l.split("\t")[14] != "NA") > 0


@pytest.mark.gpu
def test_gpu_abi_state_and_argument_errors(gpu_genome):
    from amplipy_b200.engine import AmpError, Engine
    e = Engine(ref_len=GL, n_samples=2)
    lib = e.lib
    ok = [Feature("a", "c", 1, 0, [(0, 90)])]
    n = ctypes.c_int64(0)
    assert lib.amp_annotate(e._ctx, ctypes.byref(n)) == -4                     # AMP_ERR_STATE: no features
    with pytest.raises(AmpError, match=r"\(-4\)"):
        e.set_features(0, ok)                                                  # no reference yet
    assert lib.amp_annot_host(e._ctx, None, None, None, None, None, None) == -4
    e.set_sample_reference(0, gpu_genome[:1000])
    e.set_sample_reference(1, gpu_genome)
    for bad in ([Feature("a", "c", 1, 3, [(0, 90)])], [Feature("a", "c", 0, 0, [(0, 90)])], [Feature("a", "c", 1, 0, [(50, 50)])],
                [Feature("a", "c", 1, 0, [(-1, 50)])], [Feature("a", "c", 1, 0, [(0, 1001)])], [Feature("a", "c", 1, 0, [])]):
        with pytest.raises(AmpError, match=r"\(-2\)"):
            e.set_features(0, bad)
    with pytest.raises(AmpError, match=r"\(-2\)"):
        e.set_features(2, ok)
    e.set_features(1, [Feature("a", "c", 1, 0, [(0, 1001)])])                 # the other sample is long enough
    e.set_features(0, ok)
    a = e.annotate()
    assert int(a.off[-1]) == 90 + 999
    e.set_features(0, [])                                                     # clears sample 0
    assert lib.amp_annot_host(e._ctx, None, None, None, None, None, None) == -4   # features changed since amp_annotate
    a = e.annotate()
    assert int(a.off[GL]) == 0 and int(a.off[-1]) == 999
    e.set_sample_reference(1, gpu_genome[:500])                               # now a segment ends past sample 1's reference
    with pytest.raises(AmpError, match=r"\(-2\)"):
        e.annotate()
    e.close()
