"""VCF text output of the variant records (AmpliPy.py:261-293 header, 941-952 records).

The reference writes through pysam.VariantFile / htslib; this writer emits the same header lines in the
same order and the same fields.  Text details owned by htslib (float formatting of the Float-typed
REF_FREQ, which htslib stores as float32) are restated, not verifiable offline (SURVEY.md section 8c)."""
import os
import struct
import sys

from .primers import InputError

ERROR_TEXT_FILE_EXISTS = "File already exists"
ERROR_TEXT_INVALID_VCF_EXTENSION = "Invalid variants extension (should be .vcf, .vcf.gz, or .bcf)"


def check_output_path(path):
    low = path.lower()
    if low == "stdout":
        return
    if os.path.isfile(path):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_EXISTS, path))
    if low.endswith(".bcf"):
        raise InputError("BCF output needs htslib, which this build does not link; use .vcf or .vcf.gz: %s" % path)
    if not (low.endswith(".vcf") or low.endswith(".vcf.gz")):
        raise InputError("%s: %s" % (ERROR_TEXT_INVALID_VCF_EXTENSION, path))


def header_text(contigs, version, argv):
    """``contigs``: the reference's ID, or a list of contig IDs (one ##contig line each, in that order)."""
    ids = [contigs] if isinstance(contigs, str) else list(contigs)
    lines = ["##fileformat=VCFv4.2",
             '##FILTER=<ID=PASS,Description="All filters passed">',
             "##AmpliPyVersion=%s" % version,
             "##source=%s" % " ".join(argv)] + ["##contig=<ID=%s>" % c for c in ids] + [
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
             '##INFO=<ID=DP,Number=1,Type=Integer,Description="Total Depth">',
             '##INFO=<ID=REF_DP,Number=1,Type=Integer,Description="Depth of reference base">',
             '##INFO=<ID=ALT_DP,Number=1,Type=String,Description="Depth of alternate base">',
             '##INFO=<ID=REF_FREQ,Number=1,Type=Float,Description="Frequency of reference base">',
             '##INFO=<ID=ALT_FREQ,Number=1,Type=String,Description="Frequency of alternate base">',
             "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tsample"]
    return "\n".join(lines) + "\n"


_F32 = struct.Struct("f")


def _f32(x):
    return "%g" % _F32.unpack(_F32.pack(x))[0]


def record_line(ref_genome_id, rec):
    """rec = (pos0, ref, [alts], DP, REF_DP, [ALT_DP], REF_FREQ, [ALT_FREQ], GT) from calling.variant_records.
    ALT_FREQ uses python's repr of the float64, as ','.join(str(freq)) does in AmpliPy.py:946."""
    pos0, ref, alts, dp, ref_dp, alt_dp, ref_freq, alt_freq, gt = rec
    if len(alts) == 1:          # the common case without the joins
        return "%s\t%d\t.\t%s\t%s\t.\tPASS\tDP=%d;REF_DP=%d;ALT_DP=%d;REF_FREQ=%s;ALT_FREQ=%r\tGT\t%s" % (
            ref_genome_id, pos0 + 1, ref, alts[0], dp, ref_dp, alt_dp[0], _f32(ref_freq), float(alt_freq[0]), "/".join(map(str, gt)))
    info = "DP=%d;REF_DP=%d;ALT_DP=%s;REF_FREQ=%s;ALT_FREQ=%s" % (
        dp, ref_dp, ",".join(map(str, alt_dp)), _f32(ref_freq), ",".join([repr(float(f)) for f in alt_freq]))
    return "\t".join([ref_genome_id, str(pos0 + 1), ".", ref, ",".join(alts), ".", "PASS", info, "GT", "/".join(map(str, gt))])


def write_vcf(path, contigs, version, argv, records):
    """``contigs`` = the reference's ID and ``records`` its records, or a list of contig IDs and one list of records per contig
    (written contig by contig, CHROM = the contig's ID)."""
    if isinstance(contigs, str):
        contigs, records = [contigs], [records]
    text = header_text(contigs, version, argv) + "".join(record_line(c, r) + "\n" for c, recs in zip(contigs, records) for r in recs)
    if path.lower() == "stdout":
        sys.stdout.write(text)
    elif path.lower().endswith(".gz"):
        from .alnio import bgzf_compress
        with open(path, "wb") as f:
            f.write(bgzf_compress(text.encode()))
    else:
        with open(path, "w") as f:
            f.write(text)
