"""GFF3 CDS features for the codon columns of the iVar TSV (``--gff``, DESIGN.md 3.9).

Only the host's part lives here: parsing the file and checking it.  The codon table and the translations are built on the
device (``Engine.set_features`` / ``Engine.annotate``)."""
import gzip
import os
from dataclasses import dataclass, field
from urllib.parse import unquote

from .primers import InputError

ERROR_TEXT_FILE_NOT_FOUND = "File not found"
ERROR_TEXT_INVALID_GFF_LINE = "Invalid GFF line"
ERROR_TEXT_INVALID_GFF_COORDS = "Invalid GFF start / end"
ERROR_TEXT_INVALID_GFF_STRAND = "Invalid GFF CDS strand"
ERROR_TEXT_INVALID_GFF_PHASE = "Invalid GFF CDS phase"
ERROR_TEXT_GFF_NO_ID = "GFF CDS without ID or Parent"
ERROR_TEXT_GFF_MIXED = "GFF feature with segments on different sequences or strands"
ERROR_TEXT_GFF_NO_CDS = "No CDS features in GFF file"
ERROR_TEXT_GFF_PAST_END = "GFF CDS ends past the end of its sequence"
ERROR_TEXT_GFF_SEQID_NOT_IN_FASTA = "GFF seqid is not a sequence of the reference FASTA"
ERROR_TEXT_GFF_MANY_SEQIDS = "GFF CDS rows name more than one sequence (use --multi_contig)"


@dataclass
class Feature:
    """One CDS feature: the CDS rows that share an ID (or, without one, a Parent)."""
    name: str
    seqid: str
    strand: int                                     # +1 / -1
    phase: int = 0                                  # bases skipped before the first codon (the 5'-most segment's phase)
    segments: list = field(default_factory=list)    # [(start, end)] 0-based half-open, 5' to 3'
    _phases: list = field(default_factory=list, repr=False)


def _attributes(text):
    out = {}
    for part in text.strip().split(";"):
        if "=" in part:
            k, v = part.split("=", 1)
            out[k.strip()] = unquote(v.strip())
    return out


def load_gff(path):
    """The CDS features of a GFF3 file (``.gz`` accepted) in order of first appearance, each with its segments ordered 5' to 3'
    (ascending start on '+', descending on '-').  Reading stops at ``##FASTA``; other ``#`` lines and blank lines are skipped."""
    if not os.path.isfile(path):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_NOT_FOUND, path))
    opener = gzip.open if path.lower().endswith(".gz") else open
    with opener(path, "rt") as f:
        lines = f.read().splitlines()
    feats = {}
    for l in lines:
        if l.startswith("##FASTA"):
            break
        if l.startswith("#") or not l.strip():
            continue
        parts = l.split("\t")
        if len(parts) != 9:
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_GFF_LINE, l))
        seqid, _, ftype, start, end, _, strand, phase, attrs = parts
        if ftype != "CDS":
            continue
        try:
            s, e = int(start), int(end)
        except ValueError:
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_GFF_COORDS, l))
        if s < 1 or e < s:
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_GFF_COORDS, l))
        if strand not in ("+", "-"):
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_GFF_STRAND, l))
        if phase not in ("0", "1", "2", "."):
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_GFF_PHASE, l))
        a = _attributes(attrs)
        name = a.get("ID") or a.get("Parent")
        if not name:
            raise InputError("%s: %s" % (ERROR_TEXT_GFF_NO_ID, l))
        sd = 1 if strand == "+" else -1
        ft = feats.get(name)
        if ft is None:
            ft = feats[name] = Feature(name, seqid, sd)
        elif ft.seqid != seqid or ft.strand != sd:
            raise InputError("%s: %s" % (ERROR_TEXT_GFF_MIXED, name))
        ft.segments.append((s - 1, e))
        ft._phases.append(0 if phase == "." else int(phase))
    if not feats:
        raise InputError("%s: %s" % (ERROR_TEXT_GFF_NO_CDS, path))
    out = []
    for ft in feats.values():
        order = sorted(range(len(ft.segments)), key=lambda k: ft.segments[k][0] * ft.strand)
        ft.segments = [ft.segments[k] for k in order]
        ft.phase = ft._phases[order[0]]
        ft._phases = []
        out.append(ft)
    return out


def features_by_contig(features, contigs, multi_contig):
    """The features of each contig (``contigs`` = [(ID, sequence)] in FASTA order).  With ``multi_contig`` the seqid picks the
    contig (an unknown seqid is an InputError); without it the seqid is ignored, as the BED chrom is, but the CDS rows must name
    one sequence only.  A segment that ends past its contig is an InputError."""
    out = [[] for _ in contigs]
    if multi_contig:
        index = {cid: k for k, (cid, _) in enumerate(contigs)}
        for ft in features:
            if ft.seqid not in index:
                raise InputError("%s: %s" % (ERROR_TEXT_GFF_SEQID_NOT_IN_FASTA, ft.seqid))
            out[index[ft.seqid]].append(ft)
    else:
        if len({ft.seqid for ft in features}) > 1:
            raise InputError(ERROR_TEXT_GFF_MANY_SEQIDS)
        out[0] = list(features)
    for k, (cid, seq) in enumerate(contigs):
        for ft in out[k]:
            if max(e for _, e in ft.segments) > len(seq):
                raise InputError("%s: %s (%s)" % (ERROR_TEXT_GFF_PAST_END, ft.name, cid))
    return out
