"""Primer BED loading and the per-position primer tables (host side, tiny one-off work).

Mirrors AmpliPy.py:235-258 (``load_primers``) and 174-209 (``find_overlapping_primers``); the tables
are what the trim kernel looks up per read (AmpliPy.py:450-451)."""
import os

import numpy as np

ERROR_TEXT_EMPTY_BED = "Empty BED file"
ERROR_TEXT_FILE_NOT_FOUND = "File not found"
ERROR_TEXT_INVALID_BED_LINE = "Invalid primer BED line"
ERROR_TEXT_BED_CHROM_NOT_IN_FASTA = "Primer BED chrom is not a sequence of the reference FASTA"


class InputError(Exception):
    """Carries the reference's error text; the CLI prints it the way AmpliPy.py:85-90 does."""


def _bed_rows(primer_fn):
    """4-column BED -> [(chrom, start, end)] in file order.  Any other column count is an "Invalid primer BED line", as in the
    reference (AmpliPy.py:235-258); no rows is an "Empty BED file"."""
    if not os.path.isfile(primer_fn):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_NOT_FOUND, primer_fn))
    with open(primer_fn, "r") as f:
        lines = f.read().strip().splitlines()
    rows = []
    for l in lines:
        parts = l.split("\t")
        try:
            if len(parts) != 4:
                raise ValueError
            rows.append((parts[0], int(parts[1]), int(parts[2])))
        except ValueError:
            raise InputError("%s: %s" % (ERROR_TEXT_INVALID_BED_LINE, l))
    if len(rows) == 0:
        raise InputError("%s: %s" % (ERROR_TEXT_EMPTY_BED, primer_fn))
    return rows


def load_primers(primer_fn):
    """4-column BED -> sorted [(start, end)] (AmpliPy.py:235-258); the chrom column is ignored, as in the reference."""
    return sorted((s, e) for _, s, e in _bed_rows(primer_fn))


def load_primers_by_contig(primer_fn, contig_ids):
    """4-column BED -> {contig ID: sorted [(start, end)]} for every ID of ``contig_ids`` (an empty list for a contig without
    primers); a chrom that is not one of them is an InputError."""
    out = {c: [] for c in contig_ids}
    for chrom, s, e in _bed_rows(primer_fn):
        if chrom not in out:
            raise InputError("%s: %s" % (ERROR_TEXT_BED_CHROM_NOT_IN_FASTA, chrom))
        out[chrom].append((s, e))
    for v in out.values():
        v.sort()
    return out


def find_overlapping_primers(ref_genome_length, primers, primer_pos_offset):
    """For every reference position p: over primers with start - offset <= p < end + offset,
    min(start) and max(end); -1 where no primer covers p (None in AmpliPy.py:190-191).
    Same result as the reference's sweep (174-209), computed primer by primer on numpy slices."""
    L = int(ref_genome_length)
    mn = np.full(L, np.iinfo(np.int32).max, np.int32)
    mx = np.full(L, -1, np.int32)
    off = int(primer_pos_offset)
    for s, e in primers:
        lo, hi = max(s - off, 0), min(e + off, L)
        if lo < hi:
            np.minimum(mn[lo:hi], s, out=mn[lo:hi])
            np.maximum(mx[lo:hi], e, out=mx[lo:hi])
    mn[mx < 0] = -1
    return mn, mx


def max_primer_len(primers):
    return max(e - s for s, e in primers)   # AmpliPy.py:876
