"""iVar-format outputs (DESIGN.md 3.7): the variants TSV and the IUPAC-ambiguity consensus.  AmpliPy itself has neither.

The per-allele numbers (strand and quality sums, mean qualities, Fisher p-values, IUPAC codes) are computed on the device
(``Engine.enable_qstats`` / ``process(..., qstats=True)`` / ``Engine.call_ivar``); this module only selects rows and formats.
"""
import gzip
import math
import os
from dataclasses import dataclass

import numpy as np

from .calling import FIXED_SYMS
from .primers import InputError

ERROR_TEXT_FILE_EXISTS = "File already exists"
ERROR_TEXT_INVALID_IUPAC_THRESHOLD = "IUPAC threshold must be between 0 and 1"
TSV_HEADER = ("REGION", "POS", "REF", "ALT", "REF_DP", "REF_RV", "REF_QUAL", "ALT_DP", "ALT_RV", "ALT_QUAL", "ALT_FREQ", "TOTAL_DP",
              "PVAL", "PASS", "GFF_FEATURE", "REF_CODON", "REF_AA", "ALT_CODON", "ALT_AA", "POS_AA")
PASS_PVAL = 0.05


@dataclass
class QStats:
    """Strand / quality sums of one sample (``amp_qstats_host``); the insertion arrays are in ``insertions()`` order."""
    rev: np.ndarray         # i32[6, L] increments of the count matrix from reverse-strand reads
    qsum: np.ndarray        # i64[6, L] phred qualities of the counted bases ('-' row: 0)
    ins_rev: np.ndarray     # i32[K]
    ins_qsum: np.ndarray    # i64[K] quality of each event's first inserted base
    ins_head: np.ndarray    # u8[K] 1: the allele's key is the one AmpliPy.py:735-736 builds at position 0


@dataclass
class IvarResult:
    """``amp_call_ivar`` outputs for all samples."""
    iupac: np.ndarray       # u8[S*L] IUPAC code, 0 = the reference's own consensus symbol
    fixed_mq: np.ndarray    # i32[S*L, 6] mean quality of A C G T N '-'
    fixed_pval: np.ndarray  # f64[S*L, 6] NaN = no TSV row
    ins_mq: np.ndarray      # i32[K]
    ins_pval: np.ndarray    # f64[K]


@dataclass
class Deletions:
    """Anchored deletion alleles (DESIGN.md 3.7, ``Engine.dels``), sorted by (sample, anchor, len); ``mq`` / ``pval`` are filled by
    ``Engine.call_ivar_dels`` (pval NaN = no TSV row)."""
    sample: np.ndarray      # i32[K]
    anchor: np.ndarray      # i32[K] 0-based reference position of the base before the deletion
    len: np.ndarray         # i32[K] deleted bases
    count: np.ndarray       # i32[K]
    rev: np.ndarray         # i32[K] events from reverse-strand reads
    qsum: np.ndarray        # i64[K] anchor qualities
    mq: np.ndarray = None   # i32[K] floor(qsum / count)
    pval: np.ndarray = None  # f64[K]

    def take(self, idx):
        f = lambda a: None if a is None else a[idx]
        return Deletions(f(self.sample), f(self.anchor), f(self.len), f(self.count), f(self.rev), f(self.qsum), f(self.mq), f(self.pval))


@dataclass
class Annotation:
    """``amp_annotate`` outputs (DESIGN.md 3.9): the occurrences of (sample, position) gp = sample * L + p, each a (feature, codon)
    pair the position belongs to, are entries [off[gp], off[gp + 1]), in feature order, then in spliced order."""
    L: int
    off: np.ndarray         # u32[S*L + 1]
    feat: np.ndarray        # i32[E] index of the feature in its sample's list
    pos_aa: np.ndarray      # i32[E] 1-based codon index
    codon_off: np.ndarray   # u8[E] offset of the position in the codon
    codons: np.ndarray      # u8[E, 18] REF_CODON, then ALT_CODON for A C G T N at that offset
    aas: np.ndarray         # u8[E, 6] REF_AA, then ALT_AA for A C G T N

    def columns(self, sample, p, alt, names):
        """The six annotation columns of a TSV row at position p with ALT ``alt``, one tuple per occurrence; ALT_CODON / ALT_AA
        are NA for '-' and '+' rows."""
        gp = sample * self.L + p
        out = []
        for e in range(int(self.off[gp]), int(self.off[gp + 1])):
            c, a = self.codons[e].tobytes().decode("latin-1"), self.aas[e].tobytes().decode("latin-1")
            k = "ACGTN".find(alt) if len(alt) == 1 else -1
            out.append((names[int(self.feat[e])], c[:3], a[0], c[3 + 3 * k:6 + 3 * k] if k >= 0 else "NA", a[1 + k] if k >= 0 else "NA",
                        int(self.pos_aa[e])))
        return out


def check_output_path(path):
    """The TSV refuses to overwrite, like the other outputs."""
    if path.lower() != "stdout" and os.path.isfile(path):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_EXISTS, path))


def check_iupac_threshold(t):
    if t is not None and not (0 <= t <= 1):
        raise InputError("%s: %s" % (ERROR_TEXT_INVALID_IUPAC_THRESHOLD, t))


def alt_text(sym, ref_char, head=False):
    """iVar's ALT column: a base as is, '-' as '-' + REF (a 1-bp deletion at the deleted base itself), an insertion key s as
    '+' + s[1:] (its first character is the anchor base), the key of AmpliPy.py:735-736 (``head``) as '+' + s[:-1]."""
    if sym == "-":
        return "-" + ref_char
    if len(sym) == 1 and sym in FIXED_SYMS:
        return sym
    return "+" + (sym[:-1] if head else sym[1:])


def tsv_rows(res, ins, iv, qs, ref_id, ref_seq, counts, sample=0, L=None, ann=None, names=None, dels=None):
    """The TSV rows of one sample: every allele with a p-value (count > 0, symbol != the FASTA character, freq >= min_freq, depth
    >= min_depth), in position order, then in the reference's allele order (AmpliPy.py:771).  ``L``: the sample's own reference
    length when it is shorter than the context's (a contig of a multi-record FASTA).  ``ann`` (an Annotation) and ``names`` (the
    sample's feature names): a row at a position with k >= 1 occurrences is written k times in a row, once per occurrence, with
    the six annotation columns appended.  ``dels`` (a Deletions from ``Engine.call_ivar_dels``): deletions are written as iVar
    writes them (DESIGN.md 3.7): the '-' channel gets no rows, and each anchored deletion with a p-value gets one row at its anchor,
    after the position's ranked alleles, in ascending length."""
    L = res.L if L is None else L
    base = sample * res.L
    fpv = iv.fixed_pval[base:base + L]
    del_rows = {}
    if dels is not None:
        fpv = fpv.copy()
        fpv[:, 5] = np.nan
        for k in np.flatnonzero((dels.sample == sample) & ~np.isnan(dels.pval)).tolist():
            del_rows.setdefault(int(dels.anchor[k]), []).append(k)
    ins_rows = {}
    if ins.k:
        sel = np.flatnonzero((ins.sample == sample) & ~np.isnan(iv.ins_pval[:ins.k]))
        for k in sel.tolist():
            ins_rows.setdefault(int(ins.pos[k]), []).append(k)
    pos = sorted(set(np.flatnonzero(~np.isnan(fpv).all(axis=1)).tolist()) | set(ins_rows) | set(del_rows))
    out = []
    for p in pos:
        gp = base + p
        D = int(res.depth[gp])
        ref_char = ref_seq[p]
        rch = "ACGTN".find(ref_char) if ref_char else -1
        ref_dp = int(counts[rch, p]) if rch >= 0 else 0
        ref_rv = int(qs.rev[rch, p]) if rch >= 0 else 0
        ref_q = int(iv.fixed_mq[gp, rch]) if rch >= 0 else 0
        alts = []   # (rank, ALT, count, rev, mq, pval)
        for ch in range(6):
            if not math.isnan(fpv[p, ch]):
                alts.append((int(res.fixed_rank[gp, ch]), alt_text(FIXED_SYMS[ch], ref_char), int(counts[ch, p]), int(qs.rev[ch, p]),
                             int(iv.fixed_mq[gp, ch]), float(fpv[p, ch])))
        for k in ins_rows.get(p, ()):
            alts.append((int(res.ins_rank[k]), alt_text(ins.strs[k], ref_char, bool(qs.ins_head[k])), int(ins.count[k]),
                         int(qs.ins_rev[k]), int(iv.ins_mq[k]), float(iv.ins_pval[k])))
        alts.sort(key=lambda a: a[0])
        for k in del_rows.get(p, ()):         # dels are sorted by length within a position
            n = int(dels.len[k])
            alts.append((None, "-" + ref_seq[p + 1:p + 1 + n], int(dels.count[k]), int(dels.rev[k]), int(dels.mq[k]), float(dels.pval[k])))
        for _, alt, c, rv, mq, pv in alts:
            row = (ref_id, p + 1, ref_char, alt, ref_dp, ref_rv, ref_q, c, rv, mq, c / D, D, pv, pv <= PASS_PVAL)
            cols = ann.columns(sample, p, alt, names) if ann is not None else ()
            out.extend([row + a for a in cols] if cols else [row])
    return out


def format_row(r):
    """A row of tsv_rows: 14 fields, and the six annotation columns when it has them (else NA)."""
    ref_id, pos, ref, alt, ref_dp, ref_rv, ref_q, c, rv, mq, freq, D, pv, ok = r[:14]
    ann = [str(x) for x in r[14:]] if len(r) > 14 else ["NA"] * 6
    return "\t".join([ref_id, str(pos), ref, alt, str(ref_dp), str(ref_rv), str(ref_q), str(c), str(rv), str(mq), repr(freq), str(D),
                      repr(pv), "TRUE" if ok else "FALSE"] + ann)


def write_tsv(path, rows):
    text = "\t".join(TSV_HEADER) + "\n" + "".join(format_row(r) + "\n" for r in rows)
    if path.lower() == "stdout":
        import sys
        sys.stdout.write(text)
    elif path.lower().endswith(".gz"):
        with gzip.open(path, "wt") as f:
            f.write(text)
    else:
        with open(path, "w") as f:
            f.write(text)
