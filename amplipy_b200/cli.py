"""Command line and driver with the reference's surface (AmpliPy.py:113-171 parse_args, 774-963
run_amplipy, 966-1025 dispatch): subcommands trim / variants / consensus / aio with the same flags,
defaults, validation messages and log lines.  The per-read and per-position loops run on the GPU
through the C ABI (engine.Engine); there is no CPU path."""
import argparse
import gzip
import os
import sys
from datetime import datetime

from . import alnio, calling, gff, ivar, vcf
from .primers import InputError, find_overlapping_primers, load_primers, load_primers_by_contig, max_primer_len

VERSION = "0.0.2"
DESCRIPTION = "\nAmpliPy: Python toolkit for viral amplicon sequencing\n"

# default arguments (AmpliPy.py:22-30)
DEFAULT_MIN_DEPTH_CONSENSUS = 10
DEFAULT_MIN_DEPTH_VARIANTS = 1
DEFAULT_MIN_FREQ_CONSENSUS = 0
DEFAULT_MIN_FREQ_VARIANTS = 0.03
DEFAULT_MIN_LENGTH = 30
DEFAULT_MIN_QUALITY = 20
DEFAULT_PRIMER_POS_OFFSET = 0
DEFAULT_SLIDING_WINDOW_WIDTH = 4
DEFAULT_UNKNOWN_SYMBOL = 'N'
PROGRESS_NUM_READS = 50000          # AmpliPy.py:19

# messages (AmpliPy.py:47-78)
ERROR_TEXT_FILE_NOT_FOUND = "File not found"
ERROR_TEXT_INVALID_FASTA = "Invalid FASTA file"
ERROR_TEXT_INVALID_MIN_DEPTH = "Minimum depth must be positive"
ERROR_TEXT_INVALID_MIN_FREQ = "Minimum frequency must be between 0 and 1"
ERROR_TEXT_INVALID_MIN_LENGTH = "Minimum length must be >= 1"
ERROR_TEXT_INVALID_SLIDING_WINDOW_WIDTH = "Sliding window width must be >= 1"
ERROR_TEXT_INVALID_UNKNOWN_SYMBOL_LENGTH = "Unknown symbol must be exactly 1 character"
ERROR_TEXT_MULTIPLE_REF_SEQS = "Multiple sequences in FASTA file"
ERROR_TEXT_NEGATIVE_MIN_QUALITY = "Minimum quality must be non-negative"
ERROR_TEXT_NEGATIVE_PRIMER_POS_OFFSET = "Primer position offset must be non-negative"
HELP_TEXT_CONSENSUS = "Consensus Sequence (FASTA)"
HELP_TEXT_MIN_DEPTH_CONSENSUS = "Minimum depth to call consensus"
HELP_TEXT_MIN_DEPTH_VARIANTS = "Minimum depth to call variant"
HELP_TEXT_MIN_FREQ_CONSENSUS = "Minimum frequency threshold (0-1) to call consensus"
HELP_TEXT_MIN_FREQ_VARIANTS = "Minimum frequency threshold (0-1) to call variant"
HELP_TEXT_MIN_QUAL = "Minimum quality threshold"
HELP_TEXT_PRIMER = "Primer File (BED)"
HELP_TEXT_READS_UNTRIMMED = "Untrimmed Reads (SAM/BAM)"
HELP_TEXT_READS_TRIMMED = "Trimmed Reads (SAM/BAM)"
HELP_TEXT_REFERENCE = "Reference Genome (FASTA)"
HELP_TEXT_TRIM_INCLUDE_READS_NO_PRIMER = "Include reads with no primers"
HELP_TEXT_TRIM_MIN_LENGTH = "Minimum length of read to retain after trimming"
HELP_TEXT_TRIM_PRIMER_POS_OFFSET = ("Primer position offset. Reads that occur at the specified offset positions relative to "
                                    "primer positions will also be trimmed")
HELP_TEXT_TRIM_SLIDING_WINDOW_WIDTH = "Width of sliding window (average quality of this window must be >= minimum quality threshold)"
HELP_TEXT_UNKNOWN_SYMBOL = "Character to print in regions with less than minimum coverage"
HELP_TEXT_VARIANTS = "Variant Calls (VCF)"
HELP_TEXT_TSV = "Variant Calls in iVar's TSV format, with strand counts, mean qualities and Fisher p-values (optional)"
HELP_TEXT_MULTI_CONTIG = ("Every record of the reference FASTA is a contig (e.g. the segments of a segmented virus): reads, primers "
                          "and outputs are taken per contig by name")
ERROR_TEXT_EMPTY_FASTA_RECORD = "Empty sequence in FASTA file"
ERROR_TEXT_DUPLICATE_FASTA_ID = "Duplicate sequence ID in FASTA file"
ERROR_TEXT_LENGTH_MISMATCH = "Sequence length in the alignment header differs from the reference FASTA"
ERROR_TEXT_UNKNOWN_CONTIG = "Reads on a sequence that is not in the reference FASTA"
ERROR_TEXT_UNMAPPED_NO_FLAG = "Read without a reference sequence is not flagged unmapped (flag 4)"
ERROR_TEXT_BAD_REFID = "Read reference ID outside the alignment header"
HELP_TEXT_GFF = ("GFF3 file whose CDS features fill the GFF_FEATURE / codon / amino-acid columns of the TSV (optional; needs "
                 "--output_tsv)")
ERROR_TEXT_GFF_NEEDS_TSV = "--gff needs --output_tsv"
HELP_TEXT_IVAR_DELETIONS = ("Write deletions in the TSV as iVar does: one row per deletion allele at the aligned base before it, ALT = '-' + "
                            "the deleted bases, instead of one '-' row per deleted base (optional; needs --output_tsv)")
ERROR_TEXT_DELS_NEEDS_TSV = "--ivar_deletions needs --output_tsv"
HELP_TEXT_IUPAC_THRESHOLD = ("Write IUPAC ambiguity codes: the shortest prefix of the sorted alleles whose frequencies reach this "
                             "threshold (0-1) is coded (optional; 0 = the plain consensus)")


def print_log(s='', end='\n'):
    print("[%s] %s" % (datetime.now().strftime("%Y-%m-%d %H:%M:%S"), s), end=end, file=sys.stderr)
    sys.stderr.flush()


def error(s=None):
    print_log("ERROR" if s is None else "ERROR: %s" % s)
    sys.exit(1)


def parse_args(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if len(argv) == 0:
        argv.append('-h')
    F = argparse.ArgumentDefaultsHelpFormatter
    parser = argparse.ArgumentParser(description=DESCRIPTION, formatter_class=F)
    sub = parser.add_subparsers(dest='command')

    t = sub.add_parser("trim", description=DESCRIPTION, formatter_class=F)
    t.add_argument('-i', '--input', required=False, type=str, default='stdin', help=HELP_TEXT_READS_UNTRIMMED)
    t.add_argument('-p', '--primer', required=True, type=str, help=HELP_TEXT_PRIMER)
    t.add_argument('-r', '--reference', required=True, type=str, help=HELP_TEXT_REFERENCE)
    t.add_argument('--multi_contig', action='store_true', help=HELP_TEXT_MULTI_CONTIG)
    t.add_argument('-o', '--output', required=False, type=str, default='stdout', help=HELP_TEXT_READS_TRIMMED)
    t.add_argument('-x', '--primer_pos_offset', required=False, type=int, default=DEFAULT_PRIMER_POS_OFFSET, help=HELP_TEXT_TRIM_PRIMER_POS_OFFSET)
    t.add_argument('-ml', '--min_length', required=False, type=int, default=DEFAULT_MIN_LENGTH, help=HELP_TEXT_TRIM_MIN_LENGTH)
    t.add_argument('-mq', '--min_quality', required=False, type=int, default=DEFAULT_MIN_QUALITY, help=HELP_TEXT_MIN_QUAL)
    t.add_argument('-s', '--sliding_window_width', required=False, type=int, default=DEFAULT_SLIDING_WINDOW_WIDTH, help=HELP_TEXT_TRIM_SLIDING_WINDOW_WIDTH)
    t.add_argument('-e', '--include_no_primer', action='store_true', help=HELP_TEXT_TRIM_INCLUDE_READS_NO_PRIMER)

    v = sub.add_parser("variants", description=DESCRIPTION, formatter_class=F)
    v.add_argument('-i', '--input', required=False, type=str, default='stdin', help=HELP_TEXT_READS_TRIMMED)
    v.add_argument('-r', '--reference', required=True, type=str, help=HELP_TEXT_REFERENCE)
    v.add_argument('--multi_contig', action='store_true', help=HELP_TEXT_MULTI_CONTIG)
    v.add_argument('-o', '--output', required=False, type=str, default='stdout', help=HELP_TEXT_VARIANTS)
    v.add_argument('-mq', '--min_quality', required=False, type=int, default=DEFAULT_MIN_QUALITY, help=HELP_TEXT_MIN_QUAL)
    v.add_argument('-mf', '--min_freq', required=False, type=float, default=DEFAULT_MIN_FREQ_VARIANTS, help=HELP_TEXT_MIN_FREQ_VARIANTS)
    v.add_argument('-md', '--min_depth', required=False, type=int, default=DEFAULT_MIN_DEPTH_VARIANTS, help=HELP_TEXT_MIN_DEPTH_VARIANTS)
    v.add_argument('--output_tsv', required=False, type=str, default=None, help=HELP_TEXT_TSV)
    v.add_argument('--gff', required=False, type=str, default=None, help=HELP_TEXT_GFF)
    v.add_argument('--ivar_deletions', action='store_true', help=HELP_TEXT_IVAR_DELETIONS)

    c = sub.add_parser("consensus", description=DESCRIPTION, formatter_class=F)
    c.add_argument('-i', '--input', required=False, type=str, default='stdin', help=HELP_TEXT_READS_TRIMMED)
    c.add_argument('-r', '--reference', required=True, type=str, help=HELP_TEXT_REFERENCE)
    c.add_argument('--multi_contig', action='store_true', help=HELP_TEXT_MULTI_CONTIG)
    c.add_argument('-o', '--output', required=False, type=str, default='stdout', help=HELP_TEXT_CONSENSUS)
    c.add_argument('-mq', '--min_quality', required=False, type=int, default=DEFAULT_MIN_QUALITY, help=HELP_TEXT_MIN_QUAL)
    c.add_argument('-mf', '--min_freq', required=False, type=float, default=DEFAULT_MIN_FREQ_CONSENSUS, help=HELP_TEXT_MIN_FREQ_CONSENSUS)
    c.add_argument('-md', '--min_depth', required=False, type=int, default=DEFAULT_MIN_DEPTH_CONSENSUS, help=HELP_TEXT_MIN_DEPTH_CONSENSUS)
    c.add_argument('-n', '--unknown_symbol', required=False, type=str, default=DEFAULT_UNKNOWN_SYMBOL, help=HELP_TEXT_UNKNOWN_SYMBOL)
    c.add_argument('--iupac_threshold', required=False, type=float, default=None, help=HELP_TEXT_IUPAC_THRESHOLD)

    a = sub.add_parser("aio", description=DESCRIPTION, formatter_class=F)
    a.add_argument('-i', '--input', required=False, type=str, default='stdin', help=HELP_TEXT_READS_UNTRIMMED)
    a.add_argument('-p', '--primer', required=True, type=str, help=HELP_TEXT_PRIMER)
    a.add_argument('-r', '--reference', required=True, type=str, help=HELP_TEXT_REFERENCE)
    a.add_argument('--multi_contig', action='store_true', help=HELP_TEXT_MULTI_CONTIG)
    a.add_argument('-ot', '--output_trimmed_reads', required=True, type=str, help=HELP_TEXT_READS_TRIMMED)
    a.add_argument('-ov', '--output_variants', required=True, type=str, help=HELP_TEXT_VARIANTS)
    a.add_argument('-oc', '--output_consensus', required=True, type=str, help=HELP_TEXT_CONSENSUS)
    a.add_argument('-x', '--primer_pos_offset', required=False, type=int, default=DEFAULT_PRIMER_POS_OFFSET, help=HELP_TEXT_TRIM_PRIMER_POS_OFFSET)
    a.add_argument('-ml', '--min_length', required=False, type=int, default=DEFAULT_MIN_LENGTH, help=HELP_TEXT_TRIM_MIN_LENGTH)
    a.add_argument('-mq', '--min_quality', required=False, type=int, default=DEFAULT_MIN_QUALITY, help=HELP_TEXT_MIN_QUAL)
    a.add_argument('-s', '--sliding_window_width', required=False, type=int, default=DEFAULT_SLIDING_WINDOW_WIDTH, help=HELP_TEXT_TRIM_SLIDING_WINDOW_WIDTH)
    a.add_argument('-mfc', '--min_freq_consensus', required=False, type=float, default=DEFAULT_MIN_FREQ_CONSENSUS, help=HELP_TEXT_MIN_FREQ_CONSENSUS)
    a.add_argument('-mfv', '--min_freq_variants', required=False, type=float, default=DEFAULT_MIN_FREQ_VARIANTS, help=HELP_TEXT_MIN_FREQ_VARIANTS)
    a.add_argument('-mdc', '--min_depth_consensus', required=False, type=int, default=DEFAULT_MIN_DEPTH_CONSENSUS, help=HELP_TEXT_MIN_DEPTH_CONSENSUS)
    a.add_argument('-mdv', '--min_depth_variants', required=False, type=int, default=DEFAULT_MIN_DEPTH_VARIANTS, help=HELP_TEXT_MIN_DEPTH_VARIANTS)
    a.add_argument('-n', '--unknown_symbol', required=False, type=str, default=DEFAULT_UNKNOWN_SYMBOL, help=HELP_TEXT_UNKNOWN_SYMBOL)
    a.add_argument('-e', '--include_no_primer', action='store_true', help=HELP_TEXT_TRIM_INCLUDE_READS_NO_PRIMER)
    a.add_argument('--output_tsv', required=False, type=str, default=None, help=HELP_TEXT_TSV)
    a.add_argument('--gff', required=False, type=str, default=None, help=HELP_TEXT_GFF)
    a.add_argument('--ivar_deletions', action='store_true', help=HELP_TEXT_IVAR_DELETIONS)
    a.add_argument('--iupac_threshold', required=False, type=float, default=None, help=HELP_TEXT_IUPAC_THRESHOLD)
    return parser.parse_args(argv)


def load_ref_genome(reference_fn):
    """Single-record FASTA -> (ID, sequence) (AmpliPy.py:212-232)."""
    if not os.path.isfile(reference_fn):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_NOT_FOUND, reference_fn))
    with open(reference_fn, 'r') as f:
        lines = f.read().strip().splitlines()
    if len(lines) < 2 or not lines[0].startswith('>'):
        raise InputError("%s: %s" % (ERROR_TEXT_INVALID_FASTA, reference_fn))
    ref_id = lines[0][1:].split()[0].strip()
    seq = ''.join(lines[1:])
    if '>' in seq:
        raise InputError("%s: %s" % (ERROR_TEXT_MULTIPLE_REF_SEQS, reference_fn))
    return ref_id, seq


def load_ref_genomes(reference_fn):
    """Every record of a FASTA -> [(ID, sequence)] in file order; the ID is the first whitespace token of the header, as in
    load_ref_genome.  An empty record or a repeated ID is an InputError."""
    if not os.path.isfile(reference_fn):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_NOT_FOUND, reference_fn))
    with open(reference_fn, 'r') as f:
        lines = f.read().strip().splitlines()
    if len(lines) < 2 or not lines[0].startswith('>'):
        raise InputError("%s: %s" % (ERROR_TEXT_INVALID_FASTA, reference_fn))
    recs = []
    for l in lines:
        if l.startswith('>'):
            head = l[1:].split()
            if not head:
                raise InputError("%s: %s" % (ERROR_TEXT_INVALID_FASTA, reference_fn))
            recs.append((head[0], []))
        else:
            recs[-1][1].append(l)
    out, seen = [], set()
    for rid, parts in recs:
        if rid in seen:
            raise InputError("%s: %s" % (ERROR_TEXT_DUPLICATE_FASTA_ID, rid))
        seen.add(rid)
        seq = ''.join(parts)
        if not seq:
            raise InputError("%s: %s" % (ERROR_TEXT_EMPTY_FASTA_RECORD, rid))
        out.append((rid, seq))
    return out


def header_contig_map(refs, contigs):
    """The sample (= FASTA record index) of every sequence of the alignment header (``refs`` = [(name, length)]), -2 for a
    sequence that is not in the FASTA; a length that differs from the FASTA record's is an InputError."""
    index = {rid: k for k, (rid, _) in enumerate(contigs)}
    out = []
    for name, ln in refs:
        k = index.get(name, -2)
        if k >= 0 and int(ln) != len(contigs[k][1]):
            raise InputError("%s: %s (%d vs %d)" % (ERROR_TEXT_LENGTH_MISMATCH, name, int(ln), len(contigs[k][1])))
        out.append(k)
    return out


def sam_read_contigs(aln, contigs):
    """The sample of every read of a SAM input: RNAME through the @SQ lines, or straight to the FASTA IDs when there are none;
    '*' = no contig (-1).  A read on a sequence that is not in the FASTA is an InputError naming it."""
    import numpy as np
    if aln.refs:
        m = header_contig_map(aln.refs, contigs)
        index = {name: m[r] for r, (name, _) in enumerate(aln.refs)}
    else:
        index = {rid: k for k, (rid, _) in enumerate(contigs)}
    sid = np.empty(aln.n, np.int32)
    for i, f in enumerate(aln.sam_fields):
        k = -1 if f[2] == '*' else index.get(f[2], -2)
        if k == -2:
            raise InputError("%s: %s" % (ERROR_TEXT_UNKNOWN_CONTIG, f[2]))
        sid[i] = k
    return sid


def bam_read_contigs(aln, contigs):
    """The sample of every read of a BAM input decoded on the host: its refID through header_contig_map."""
    import numpy as np
    m = np.array(header_contig_map(aln.refs, contigs) + [-1], np.int32)
    if aln.n == 0:
        return np.zeros(0, np.int32)
    rid = aln.bam_buf[aln.bam_rec_off[:, None] + 4 + np.arange(4)].copy().view(np.int32).ravel()
    if ((rid < -1) | (rid >= len(aln.refs))).any():
        raise InputError(ERROR_TEXT_BAD_REFID)
    sid = m[rid]
    if (sid == -2).any():
        raise InputError("%s: %s" % (ERROR_TEXT_UNKNOWN_CONTIG, aln.refs[int(rid[np.flatnonzero(sid == -2)[0]])][0]))
    return sid


def check_contig_plan(plan, refs=None, ref_map=None):
    """InputError for what amp_contig_plan_* flags: reads on sequences that are not in the FASTA (named), reads without a
    reference that are not flagged unmapped, refIDs outside the header."""
    from .engine import CONTIG_E_BADID, CONTIG_E_NOFLAG4, CONTIG_E_UNKNOWN
    if plan.errors & CONTIG_E_UNKNOWN:
        names = [refs[r][0] for r in range(len(refs)) if ref_map[r] == -2 and plan.ref_reads[r]]
        raise InputError("%s: %s" % (ERROR_TEXT_UNKNOWN_CONTIG, ", ".join(names)))
    if plan.errors & CONTIG_E_NOFLAG4:
        raise InputError(ERROR_TEXT_UNMAPPED_NO_FLAG)
    if plan.errors & CONTIG_E_BADID:
        raise InputError(ERROR_TEXT_BAD_REFID)


def dels_slots(sum_cigar_ops):
    """Slots of the anchored deletion table for a batch of ``sum_cigar_ops`` CIGAR ops: every allele comes from a D op of the input
    (trimming merges or drops D ops, it adds none), so twice their total, rounded up to a power of two, never fills."""
    return max(1024, 1 << int(2 * max(int(sum_cigar_ops), 1) - 1).bit_length())


def run_amplipy(untrimmed_reads_fn=None, primer_fn=None, reference_fn=None, trimmed_reads_fn=None, variants_fn=None,
                consensus_fn=None, primer_pos_offset=None, min_length=None, min_quality=None, sliding_window_width=None,
                min_freq_consensus=None, min_freq_variants=None, min_depth_consensus=None, min_depth_variants=None,
                unknown_symbol=None, include_no_primer=None, run_trim=False, run_variants=False, run_consensus=False,
                argv=None, device=0, tsv_fn=None, iupac_threshold=None, multi_contig=False, gff_fn=None, ivar_deletions=False):
    """Same keyword arguments and behaviour as the reference's run_amplipy (AmpliPy.py:774-963).  Additions of this
    project: ``tsv_fn`` (with run_variants) also writes the variants in iVar's TSV format, ``iupac_threshold`` (with
    run_consensus) writes IUPAC ambiguity codes into the consensus (DESIGN.md 3.7), ``multi_contig`` takes every record of the
    reference FASTA as a contig (DESIGN.md 3.8), ``gff_fn`` (with ``tsv_fn``) fills the TSV's codon columns from the CDS
    features of a GFF3 file (DESIGN.md 3.9), ``ivar_deletions`` (with ``tsv_fn``) writes the TSV's deletions as iVar does, one
    row per anchored deletion allele (DESIGN.md 3.7)."""
    argv = list(sys.argv if argv is None else argv)
    try:
        return _run(untrimmed_reads_fn, primer_fn, reference_fn, trimmed_reads_fn, variants_fn, consensus_fn, primer_pos_offset,
                    min_length, min_quality, sliding_window_width, min_freq_consensus, min_freq_variants, min_depth_consensus,
                    min_depth_variants, unknown_symbol, include_no_primer, run_trim, run_variants, run_consensus, argv, device,
                    tsv_fn if run_variants else None, iupac_threshold if run_consensus else None, multi_contig,
                    gff_fn if run_variants else None, bool(ivar_deletions) and run_variants)
    except InputError as e:
        error(str(e))


def _run(untrimmed_reads_fn, primer_fn, reference_fn, trimmed_reads_fn, variants_fn, consensus_fn, primer_pos_offset, min_length,
         min_quality, sliding_window_width, min_freq_consensus, min_freq_variants, min_depth_consensus, min_depth_variants,
         unknown_symbol, include_no_primer, run_trim, run_variants, run_consensus, argv, device, tsv_fn=None, iupac_threshold=None,
         multi_contig=False, gff_fn=None, ivar_deletions=False):
    # validity checks (AmpliPy.py:837-854)
    if primer_pos_offset is not None and primer_pos_offset < 0:
        error("%s: %s" % (ERROR_TEXT_NEGATIVE_PRIMER_POS_OFFSET, primer_pos_offset))
    if min_length is not None and min_length < 1:
        error("%s: %s" % (ERROR_TEXT_INVALID_MIN_LENGTH, min_length))
    if min_quality is not None and min_quality < 0:
        error("%s: %s" % (ERROR_TEXT_NEGATIVE_MIN_QUALITY, min_quality))
    if sliding_window_width is not None and sliding_window_width < 1:
        error("%s: %s" % (ERROR_TEXT_INVALID_SLIDING_WINDOW_WIDTH, sliding_window_width))
    if min_freq_consensus is not None and (min_freq_consensus < 0 or min_freq_consensus > 1):
        error("%s: %s" % (ERROR_TEXT_INVALID_MIN_FREQ, min_freq_consensus))
    if min_freq_variants is not None and (min_freq_variants < 0 or min_freq_variants > 1):
        error("%s: %s" % (ERROR_TEXT_INVALID_MIN_FREQ, min_freq_variants))
    if min_depth_consensus is not None and min_depth_consensus < 0:
        error("%s: %s" % (ERROR_TEXT_INVALID_MIN_DEPTH, min_depth_consensus))
    if min_depth_variants is not None and min_depth_variants < 0:
        error("%s: %s" % (ERROR_TEXT_INVALID_MIN_DEPTH, min_depth_variants))
    if unknown_symbol is not None and len(unknown_symbol) != 1:
        error("%s: %s" % (ERROR_TEXT_INVALID_UNKNOWN_SYMBOL_LENGTH, unknown_symbol))
    if iupac_threshold is not None and not (0 <= iupac_threshold <= 1):
        error("%s: %s" % (ivar.ERROR_TEXT_INVALID_IUPAC_THRESHOLD, iupac_threshold))
    if gff_fn is not None and tsv_fn is None:
        error(ERROR_TEXT_GFF_NEEDS_TSV)
    if ivar_deletions and tsv_fn is None:
        error(ERROR_TEXT_DELS_NEEDS_TSV)

    # mode banner (AmpliPy.py:857-866)
    if not (run_trim or run_variants or run_consensus):
        error("Not running any of the AmpliPy operations")
    if run_trim and not (run_variants or run_consensus):
        print_log("Executing AmpliPy Trim (v%s)" % VERSION)
    elif run_variants and not (run_trim or run_consensus):
        print_log("Executing AmpliPy Variants (v%s)" % VERSION)
    elif run_consensus and not (run_trim or run_variants):
        print_log("Executing AmpliPy Consensus (v%s)" % VERSION)
    else:
        print_log("Executing AmpliPy All-In-One (v%s)" % VERSION)

    print_log("Loading reference genome: %s" % reference_fn)
    if multi_contig:
        return _run_contigs(untrimmed_reads_fn, primer_fn, reference_fn, trimmed_reads_fn, variants_fn, consensus_fn, primer_pos_offset,
                            min_length, min_quality, sliding_window_width, min_freq_consensus, min_freq_variants, min_depth_consensus,
                            min_depth_variants, unknown_symbol, include_no_primer, run_trim, run_variants, run_consensus, argv, device,
                            tsv_fn, iupac_threshold, gff_fn, ivar_deletions)
    ref_id, ref_seq = load_ref_genome(reference_fn)
    L = len(ref_seq)
    tables, mpl = None, 0
    if primer_fn is not None:
        print_log("Loading primers: %s" % primer_fn)
        primers = load_primers(primer_fn)
        mpl = max_primer_len(primers)
        print_log("Precalculating overlapping primers...")
        tables = find_overlapping_primers(L, primers, primer_pos_offset)
    in_fn = untrimmed_reads_fn if run_trim else trimmed_reads_fn
    if run_trim:
        print_log("Input untrimmed SAM/BAM: %s" % untrimmed_reads_fn)
        print_log("Output trimmed SAM/BAM: %s" % trimmed_reads_fn)
        alnio.check_output_path(trimmed_reads_fn)
    else:
        print_log("Input trimmed SAM/BAM: %s" % trimmed_reads_fn)
    if variants_fn is not None:
        print_log("Output variants VCF: %s" % variants_fn)
        vcf.check_output_path(variants_fn)
    if tsv_fn is not None:
        print_log("Output variants TSV: %s" % tsv_fn)
        ivar.check_output_path(tsv_fn)
    features = None
    if gff_fn is not None:
        print_log("Loading GFF: %s" % gff_fn)
        features = gff.features_by_contig(gff.load_gff(gff_fn), [(ref_id, ref_seq)], False)[0]
    import threading
    import time as _time
    tm = {}
    from .engine import AmpError, Engine, TrimResult

    qstats = tsv_fn is not None      # the strand / quality pass runs only for the TSV

    def make_engine(indel_rich):
        e = Engine(ref_len=L, primer_tables=tables, max_primer_len=mpl,
                   min_quality=DEFAULT_MIN_QUALITY if min_quality is None else min_quality,
                   sliding_window_width=DEFAULT_SLIDING_WINDOW_WIDTH if sliding_window_width is None else sliding_window_width,
                   min_length=DEFAULT_MIN_LENGTH if min_length is None else min_length,
                   include_no_primer=bool(include_no_primer), device=device,
                   ins_slots=(1 << 24) if indel_rich else 0, ins_arena_bytes=(1 << 30) if indel_rich else 0)
        if qstats or iupac_threshold is not None:
            e.enable_qstats()
        return e
    pile = run_variants or run_consensus
    _t = _time.perf_counter()
    aln = eng = trim = None
    n_reads = 0
    if (in_fn.lower().endswith(".bam") and os.path.isfile(in_fn) and not os.environ.get("AMPLIPY_HOST_DECODE") and
            hasattr(Engine, "decode_bam")):
        # BAM: the compressed file goes to the GPU as it is and is decoded there (amp_bam_decode_host); the host inflates it too,
        # at the same time, only when the records are needed for the trimmed output
        with open(in_fn, "rb") as f:
            raw = f.read()
        layout = alnio.bam_layout(raw)
        box = {}
        host = None
        # BAM in -> BAM out: the trimmed records are rebuilt and compressed on the device as well (amp_decoded_write_bam), unless a
        # zlib level is asked for (AMPLIPY_BAM_LEVEL; 6 = what htslib writes)
        dev_bam_out = (run_trim and trimmed_reads_fn.lower().endswith(".bam") and "AMPLIPY_BAM_LEVEL" not in os.environ and
                       hasattr(Engine, "decoded_write_bam"))
        if run_trim and not dev_bam_out:
            def _host_decode():
                try:
                    box["aln"] = alnio._read_bam(raw)
                except BaseException as e:
                    box["err"] = e
            host = threading.Thread(target=_host_decode)
            host.start()
        out_header = alnio.header_with_pg(layout["header_text"], argv) if run_trim else None
        eng = make_engine(layout["ops_per_read"] > 8)
        print_log("Processing reads...")
        try:
            info = eng.decode_bam(raw, layout)
            if ivar_deletions:
                eng.enable_dels(dels_slots(info["sum_cig"]))
            outs = eng.process_decoded(trim=run_trim, pileup=pile, download=not dev_bam_out, **({"qstats": True} if qstats else {}))
            n_reads = info["n"]
        except AmpError:
            eng.close()
            eng = None                       # e.g. records straddling BGZF blocks (not written by htslib): host decoder below
            dev_bam_out = False
        tm["gpu_decode_process"] = _time.perf_counter() - _t
        if host is not None:
            host.join()
            if "err" in box:
                raise box["err"]
            aln = box["aln"]
            if eng is not None:
                trim = TrimResult(aln.batch, *outs)
        tm["decode"] = _time.perf_counter() - _t
        if eng is not None:
            eng.raise_on_device_errors()
    else:
        dev_bam_out = False
    if eng is None:
        aln = aln or alnio.read_alignments(in_fn)
        tm["decode"] = _time.perf_counter() - _t
        out_header = alnio.header_with_pg(aln.header_text, argv) if run_trim else None
        indel_rich = aln.n and (aln.batch.cigar.size / aln.n) > 8
        eng = make_engine(indel_rich)
        if ivar_deletions:
            eng.enable_dels(dels_slots(aln.batch.cigar.size))
        print_log("Processing reads...")
        _t = _time.perf_counter()
        trim = eng.process(aln.batch, trim=run_trim, pileup=pile, **({"qstats": True} if qstats else {}))
        eng.raise_on_device_errors()
        tm["gpu_process"] = _time.perf_counter() - _t
        n_reads = aln.n
    # the reference reports its progress every PROGRESS_NUM_READS reads of its loop (AmpliPy.py:19, 898-899); the reads
    # are processed as one batch here, so the same lines are written once the batch is through
    for k in range(PROGRESS_NUM_READS, n_reads, PROGRESS_NUM_READS):
        print_log("Processed %d reads..." % k)
    writer = None
    if run_trim:
        # the trimmed reads are encoded (record rewrite + BGZF deflate, both outside the GIL) while calling and the text outputs run
        def _write():
            t0 = _time.perf_counter()
            try:
                if dev_bam_out:
                    data, _ = eng.decoded_write_bam(alnio._bam_header_bytes(out_header, layout["refs"]))
                    with open(trimmed_reads_fn, "wb") as f:
                        f.write(data)
                else:
                    # BGZF deflate on the GPU unless a zlib level is asked for
                    on_gpu = "AMPLIPY_BAM_LEVEL" not in os.environ and hasattr(eng, "bgzf_deflate")
                    alnio.write_alignments(trimmed_reads_fn, aln, out_header, trim, deflater=eng.bgzf_deflate if on_gpu else None)
            except BaseException as e:      # re-raised on the main thread
                tm["_write_error"] = e
            tm["encode_bam"] = _time.perf_counter() - t0
        writer = threading.Thread(target=_write)
        writer.start()
    _t = _time.perf_counter()
    if pile:
        counts = eng.counts()
        ins = eng.insertions()
        res = eng.call(ref_seq,
                       DEFAULT_MIN_DEPTH_CONSENSUS if min_depth_consensus is None else min_depth_consensus,
                       DEFAULT_MIN_FREQ_CONSENSUS if min_freq_consensus is None else min_freq_consensus,
                       DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                       DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants)
        if run_variants:
            vcf.write_vcf(variants_fn, ref_id, VERSION, argv, calling.variant_records(res, ins, ref_seq, counts))
        if tsv_fn is not None:
            iv = eng.call_ivar(DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                               DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants)
            ann = names = None
            if features is not None:
                eng.set_features(0, features)     # after call: the context holds the reference now
                ann, names = eng.annotate(), [f.name for f in features]
            dels = eng.call_ivar_dels(DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                                      DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants) if ivar_deletions else None
            ivar.write_tsv(tsv_fn, ivar.tsv_rows(res, ins, iv, eng.qstats(0), ref_id, ref_seq, counts, ann=ann, names=names, dels=dels))
        iupac = None
        if iupac_threshold is not None:
            iupac = eng.call_ivar(DEFAULT_MIN_DEPTH_CONSENSUS if min_depth_consensus is None else min_depth_consensus,
                                  DEFAULT_MIN_FREQ_CONSENSUS if min_freq_consensus is None else min_freq_consensus,
                                  iupac_threshold).iupac
        if run_consensus:
            text = '>sample\n%s\n' % calling.consensus_string(res, ins, 0, unknown_symbol, iupac=iupac)
            if consensus_fn.lower() == 'stdout':
                sys.stdout.write(text)
            elif consensus_fn.lower().endswith('.gz'):
                with gzip.open(consensus_fn, 'wt') as f:
                    f.write(text)
            else:
                with open(consensus_fn, 'w') as f:
                    f.write(text)
    tm["call_and_text"] = _time.perf_counter() - _t
    if writer is not None:
        writer.join()
        if "_write_error" in tm:
            raise tm.pop("_write_error")
    if os.environ.get("AMP_CLI_TIMINGS"):      # bench.py's file-to-file leg: where the wall time went
        import json
        with open(os.environ["AMP_CLI_TIMINGS"], "w") as f:
            json.dump({k: round(v, 4) for k, v in tm.items()}, f)
    print_log("Finished Processing %d reads" % max(n_reads - 1, 0))
    return eng


def _run_contigs(untrimmed_reads_fn, primer_fn, reference_fn, trimmed_reads_fn, variants_fn, consensus_fn, primer_pos_offset, min_length,
                 min_quality, sliding_window_width, min_freq_consensus, min_freq_variants, min_depth_consensus, min_depth_variants,
                 unknown_symbol, include_no_primer, run_trim, run_variants, run_consensus, argv, device, tsv_fn, iupac_threshold, gff_fn=None,
                 ivar_deletions=False):
    """_run with --multi_contig (DESIGN.md 3.8): contig k of the FASTA is sample k of one context, with the BED rows of its chrom as
    its scheme and its own length; reads go to the contig their reference names.  Outputs follow the FASTA's record order."""
    contigs = load_ref_genomes(reference_fn)
    ids = [c[0] for c in contigs]
    lens = [len(c[1]) for c in contigs]
    schemes = {c: [] for c in ids}
    if primer_fn is not None:
        print_log("Loading primers: %s" % primer_fn)
        schemes = load_primers_by_contig(primer_fn, ids)
    in_fn = untrimmed_reads_fn if run_trim else trimmed_reads_fn
    if run_trim:
        print_log("Input untrimmed SAM/BAM: %s" % untrimmed_reads_fn)
        print_log("Output trimmed SAM/BAM: %s" % trimmed_reads_fn)
        alnio.check_output_path(trimmed_reads_fn)
    else:
        print_log("Input trimmed SAM/BAM: %s" % trimmed_reads_fn)
    if variants_fn is not None:
        print_log("Output variants VCF: %s" % variants_fn)
        vcf.check_output_path(variants_fn)
    if tsv_fn is not None:
        print_log("Output variants TSV: %s" % tsv_fn)
        ivar.check_output_path(tsv_fn)
    features = None
    if gff_fn is not None:
        print_log("Loading GFF: %s" % gff_fn)
        features = gff.features_by_contig(gff.load_gff(gff_fn), contigs, True)
    from .engine import AmpError, ContigError, Engine, TrimResult
    qstats = tsv_fn is not None
    pile = run_variants or run_consensus

    def make_engine(indel_rich):
        e = Engine(ref_len=max(lens), n_samples=len(contigs),
                   min_quality=DEFAULT_MIN_QUALITY if min_quality is None else min_quality,
                   sliding_window_width=DEFAULT_SLIDING_WINDOW_WIDTH if sliding_window_width is None else sliding_window_width,
                   min_length=DEFAULT_MIN_LENGTH if min_length is None else min_length,
                   include_no_primer=bool(include_no_primer), device=device,
                   ins_slots=(1 << 24) if indel_rich else 0, ins_arena_bytes=(1 << 30) if indel_rich else 0)
        for k, (cid, seq) in enumerate(contigs):
            # every contig gets a scheme, empty without primers: the coordinate checks then use the contig's own length
            e.set_scheme(k, schemes[cid], 0 if primer_pos_offset is None else primer_pos_offset, ref_len=len(seq))
            e.set_sample_reference(k, seq)
        if qstats or iupac_threshold is not None:
            e.enable_qstats()
        return e
    mode = dict(trim=run_trim, pileup=pile, qstats=qstats)
    eng = aln = trim = None
    dev_bam_out = False
    if in_fn.lower().endswith(".bam") and os.path.isfile(in_fn) and not os.environ.get("AMPLIPY_HOST_DECODE"):
        with open(in_fn, "rb") as f:
            raw = f.read()
        layout = alnio.bam_layout(raw)
        ref_map = header_contig_map(layout["refs"], contigs)
        out_header = alnio.header_with_pg(layout["header_text"], argv) if run_trim else None
        dev_bam_out = run_trim and trimmed_reads_fn.lower().endswith(".bam") and "AMPLIPY_BAM_LEVEL" not in os.environ
        eng = make_engine(layout["ops_per_read"] > 8)
        print_log("Processing reads...")
        try:
            info = eng.decode_bam(raw, layout)
        except AmpError:
            eng.close()
            eng = None                       # e.g. records straddling BGZF blocks (not written by htslib): host decoder below
            dev_bam_out = False
        if eng is not None:
            check_contig_plan(eng.contig_plan_decoded(ref_map), layout["refs"], ref_map)
            if ivar_deletions:
                eng.enable_dels(dels_slots(info["sum_cig"]))
            outs = eng.process_decoded_contigs(download=not dev_bam_out, **mode)
            eng.raise_on_device_errors()
            n_reads = info["n"]
            if run_trim and not dev_bam_out:
                aln = alnio._read_bam(raw)
                trim = TrimResult(aln.batch, *outs)
    if eng is None:
        aln = alnio.read_alignments(in_fn)
        out_header = alnio.header_with_pg(aln.header_text, argv) if run_trim else None
        sid = sam_read_contigs(aln, contigs) if aln.fmt == "sam" else bam_read_contigs(aln, contigs)
        eng = make_engine(aln.n and (aln.batch.cigar.size / aln.n) > 8)
        if ivar_deletions:
            eng.enable_dels(dels_slots(aln.batch.cigar.size))
        print_log("Processing reads...")
        try:
            trim = eng.process_contigs(aln.batch, sid, **mode)
        except ContigError as e:
            check_contig_plan(e.plan)
            raise
        eng.raise_on_device_errors()
        n_reads = aln.n
    for k in range(PROGRESS_NUM_READS, n_reads, PROGRESS_NUM_READS):
        print_log("Processed %d reads..." % k)
    if run_trim:
        if dev_bam_out:
            data, _ = eng.decoded_write_bam(alnio._bam_header_bytes(out_header, layout["refs"]))
            with open(trimmed_reads_fn, "wb") as f:
                f.write(data)
        else:
            on_gpu = "AMPLIPY_BAM_LEVEL" not in os.environ
            alnio.write_alignments(trimmed_reads_fn, aln, out_header, trim, deflater=eng.bgzf_deflate if on_gpu else None)
    if pile:
        counts = [eng.counts(k) for k in range(len(contigs))]
        ins = eng.insertions()
        res = eng.call(None,
                       DEFAULT_MIN_DEPTH_CONSENSUS if min_depth_consensus is None else min_depth_consensus,
                       DEFAULT_MIN_FREQ_CONSENSUS if min_freq_consensus is None else min_freq_consensus,
                       DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                       DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants)
        if run_variants:
            vcf.write_vcf(variants_fn, ids, VERSION, argv, [calling.variant_records(res, ins, seq, counts[k], k, L=len(seq))
                                                            for k, (_, seq) in enumerate(contigs)])
        if tsv_fn is not None:
            iv = eng.call_ivar(DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                               DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants)
            ann = None
            if features is not None:
                for k, fk in enumerate(features):
                    eng.set_features(k, fk)
                ann = eng.annotate()
            dels = eng.call_ivar_dels(DEFAULT_MIN_DEPTH_VARIANTS if min_depth_variants is None else min_depth_variants,
                                      DEFAULT_MIN_FREQ_VARIANTS if min_freq_variants is None else min_freq_variants) if ivar_deletions else None
            ivar.write_tsv(tsv_fn, [r for k, (cid, seq) in enumerate(contigs)
                                    for r in ivar.tsv_rows(res, ins, iv, eng.qstats(k), cid, seq, counts[k], k, L=len(seq), ann=ann,
                                                           names=[f.name for f in features[k]] if features is not None else None,
                                                           dels=dels)])
        iupac = None
        if iupac_threshold is not None:
            iupac = eng.call_ivar(DEFAULT_MIN_DEPTH_CONSENSUS if min_depth_consensus is None else min_depth_consensus,
                                  DEFAULT_MIN_FREQ_CONSENSUS if min_freq_consensus is None else min_freq_consensus,
                                  iupac_threshold).iupac
        if run_consensus:
            # one record per contig, headed by its ID (a repeated '>sample' would make the IDs ambiguous)
            text = "".join('>%s\n%s\n' % (cid, calling.consensus_string(res, ins, k, unknown_symbol, iupac=iupac, L=len(seq)))
                           for k, (cid, seq) in enumerate(contigs))
            if consensus_fn.lower() == 'stdout':
                sys.stdout.write(text)
            elif consensus_fn.lower().endswith('.gz'):
                with gzip.open(consensus_fn, 'wt') as f:
                    f.write(text)
            else:
                with open(consensus_fn, 'w') as f:
                    f.write(text)
    print_log("Finished Processing %d reads" % max(n_reads - 1, 0))
    return eng


def main(argv=None):
    args = parse_args(argv)
    full_argv = list(sys.argv) if argv is None else ["AmpliPy.py"] + list(argv)
    if args.command == 'trim':
        run_amplipy(untrimmed_reads_fn=args.input, primer_fn=args.primer, reference_fn=args.reference,
                    trimmed_reads_fn=args.output, primer_pos_offset=args.primer_pos_offset, min_length=args.min_length,
                    min_quality=args.min_quality, sliding_window_width=args.sliding_window_width,
                    include_no_primer=args.include_no_primer, run_trim=True, argv=full_argv, multi_contig=args.multi_contig)
    elif args.command == 'variants':
        run_amplipy(trimmed_reads_fn=args.input, reference_fn=args.reference, variants_fn=args.output,
                    min_quality=args.min_quality, min_freq_variants=args.min_freq, min_depth_variants=args.min_depth,
                    run_variants=True, argv=full_argv, tsv_fn=args.output_tsv, multi_contig=args.multi_contig, gff_fn=args.gff,
                    ivar_deletions=args.ivar_deletions)
    elif args.command == 'consensus':
        run_amplipy(trimmed_reads_fn=args.input, reference_fn=args.reference, consensus_fn=args.output,
                    min_quality=args.min_quality, min_freq_consensus=args.min_freq, min_depth_consensus=args.min_depth,
                    unknown_symbol=args.unknown_symbol, run_consensus=True, argv=full_argv, iupac_threshold=args.iupac_threshold,
                    multi_contig=args.multi_contig)
    elif args.command == 'aio':
        run_amplipy(untrimmed_reads_fn=args.input, primer_fn=args.primer, reference_fn=args.reference,
                    trimmed_reads_fn=args.output_trimmed_reads, variants_fn=args.output_variants,
                    consensus_fn=args.output_consensus, primer_pos_offset=args.primer_pos_offset, min_length=args.min_length,
                    min_quality=args.min_quality, sliding_window_width=args.sliding_window_width,
                    min_freq_consensus=args.min_freq_consensus, min_freq_variants=args.min_freq_variants,
                    min_depth_consensus=args.min_depth_consensus, min_depth_variants=args.min_depth_variants,
                    unknown_symbol=args.unknown_symbol, include_no_primer=args.include_no_primer, run_trim=True,
                    run_variants=True, run_consensus=True, argv=full_argv, tsv_fn=args.output_tsv,
                    iupac_threshold=args.iupac_threshold, multi_contig=args.multi_contig, gff_fn=args.gff,
                    ivar_deletions=args.ivar_deletions)


if __name__ == "__main__":
    main()
