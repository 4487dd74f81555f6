"""SAM / BAM input and output around the batch kernels.

Replaces the pysam surface the reference uses for I/O (AmpliPy.py:296-360 open + @PG header, 896 record
iteration, 911 ``out_aln.write``) with: whole-file decode into one struct-of-arrays ``ReadBatch``
(multi-threaded BGZF inflate + record scatter in ``csrc/amp_hostio.cpp``), and a writer that re-emits
the kept reads with only ``pos`` / ``bin`` / CIGAR changed -- everything else byte for byte.
"""
import ctypes
import os
import sys

import numpy as np

from .batch import CIGAR_CHARS, ReadBatch, cigar_string, pack_seq, parse_cigar
from .primers import InputError

ERROR_TEXT_FILE_EXISTS = "File already exists"
ERROR_TEXT_FILE_NOT_FOUND = "File not found"
ERROR_TEXT_INVALID_READ_EXTENSION = "Invalid read mapping extension (should be .sam or .bam)"
VERSION = "0.0.2"   # AmpliPy.py:17 -- recorded in the @PG line exactly as the reference does

_HERE = os.path.dirname(os.path.abspath(__file__))
_HOSTIO = os.path.join(_HERE, "csrc", "libamplipy_hostio.so")
_lib = None


def hostio():
    global _lib
    if _lib is None:
        if not os.path.isfile(_HOSTIO):
            from . import build
            build.build_hostio()
        lib = ctypes.CDLL(_HOSTIO)
        lib.amp_bgzf_scan.restype = ctypes.c_longlong
        lib.amp_bam_scan.restype = ctypes.c_longlong
        lib.amp_bgzf_bound.restype = ctypes.c_longlong
        lib.amp_bgzf_deflate.restype = ctypes.c_longlong
        lib.amp_bam_rewrite.restype = ctypes.c_longlong
        lib.amp_bgzf_deflate_blocks.restype = ctypes.c_longlong
        lib.amp_bgzf_plan.restype = ctypes.c_longlong
        lib.amp_bam_serialize.restype = ctypes.c_longlong
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _ll(v):
    return ctypes.c_longlong(int(v))


# ------------------------------------------------------------------------------------------- BGZF
def bgzf_decompress(raw, threads=0):
    """bytes of a BGZF file -> uint8 array with the concatenated payload (parallel over blocks)."""
    lib = hostio()
    src = np.frombuffer(raw, dtype=np.uint8)
    n = lib.amp_bgzf_scan(_p(src), _ll(src.size), None, None, _ll(0))
    if n < 0:
        raise InputError("Invalid BGZF stream")
    in_off = np.empty(n, np.int64)
    out_len = np.empty(n, np.uint32)
    lib.amp_bgzf_scan(_p(src), _ll(src.size), _p(in_off), _p(out_len), _ll(n))
    out_off = np.zeros(n + 1, np.int64)
    np.cumsum(out_len, out=out_off[1:])
    out = np.empty(int(out_off[-1]) + 16, np.uint8)
    if lib.amp_bgzf_inflate(_p(src), _p(in_off), _p(out_len), _p(out_off), _ll(n), _ll(src.size), _p(out), threads):
        raise InputError("Corrupt BGZF block")
    return out[:int(out_off[-1])]


def bgzf_blocks(raw):
    """Block table of a BGZF file: {"in_off": int64[n] start of every block, "out_len": uint32[n] its ISIZE}."""
    lib = hostio()
    src = np.frombuffer(raw, dtype=np.uint8)
    n = lib.amp_bgzf_scan(_p(src), _ll(src.size), None, None, _ll(0))
    if n < 0:
        raise InputError("Invalid BGZF stream")
    in_off = np.empty(n, np.int64)
    out_len = np.empty(n, np.uint32)
    lib.amp_bgzf_scan(_p(src), _ll(src.size), _p(in_off), _p(out_len), _ll(n))
    return {"in_off": in_off, "out_len": out_len}


def bam_layout(raw):
    """What the device-side decoder needs from the host, without inflating the records: the BGZF block table, the BAM header
    (text + reference list, inflated from the first block(s)) and the offset of the first record in the inflated stream."""
    import zlib
    blocks = bgzf_blocks(raw)
    in_off, out_len = blocks["in_off"], blocks["out_len"]
    mv = memoryview(raw)
    hdr = bytearray()
    k = 0

    def more():
        nonlocal k
        if k >= len(in_off):
            raise InputError("Invalid BAM file")
        a = int(in_off[k]); e = int(in_off[k + 1]) if k + 1 < len(in_off) else len(raw)
        xlen = int(mv[a + 10]) | (int(mv[a + 11]) << 8)
        try:
            hdr.extend(zlib.decompress(bytes(mv[a + 12 + xlen:e - 8]), -15))
        except zlib.error:
            raise InputError("Corrupt BGZF block")
        k += 1

    def need(n):
        while len(hdr) < n:
            more()
    need(12)
    if bytes(hdr[:4]) != b"BAM\x01":
        raise InputError("Invalid BAM file")
    l_text = int.from_bytes(hdr[4:8], "little", signed=True)
    if l_text < 0:
        raise InputError("Invalid BAM file")
    need(12 + l_text)
    header_text = bytes(hdr[8:8 + l_text]).split(b"\0", 1)[0].decode()
    p = 8 + l_text
    n_ref = int.from_bytes(hdr[p:p + 4], "little", signed=True); p += 4
    refs = []
    for _ in range(max(n_ref, 0)):
        need(p + 4)
        l_name = int.from_bytes(hdr[p:p + 4], "little", signed=True); p += 4
        if l_name < 1:
            raise InputError("Invalid BAM file")
        need(p + l_name + 4)
        name = bytes(hdr[p:p + l_name - 1]).decode(); p += l_name
        refs.append((name, int.from_bytes(hdr[p:p + 4], "little", signed=True))); p += 4
    # a look at the first records (CIGAR ops per read): callers size the insertion table for indel-rich data before decoding
    ops_per_read = 0.0
    try:
        while len(hdr) < p + 36 and k < len(in_off):
            more()
        q, nrec, nops = p, 0, 0
        while q + 36 <= len(hdr) and nrec < 256:
            bs = int.from_bytes(hdr[q:q + 4], "little")
            if bs < 32 or q + 4 + bs > len(hdr):
                break
            nops += int.from_bytes(hdr[q + 16:q + 18], "little"); nrec += 1
            q += 4 + bs
        ops_per_read = nops / nrec if nrec else 0.0
    except InputError:
        pass
    return {"in_off": in_off, "out_len": out_len, "body_off": p, "header_text": header_text, "refs": refs,
            "ops_per_read": ops_per_read}


def bgzf_compress_units(data, bounds, level=6, threads=0, deflater=None):
    """BGZF the way htslib lays a BAM out: a block holds whole units (``bounds`` = sorted cut points from 0 to len(data), e.g.
    header end + record starts) -- a record never straddles a block boundary (bgzf_flush_try in htslib's bam_write1).
    ``deflater(data, block_starts)``: compress the planned blocks elsewhere (Engine.bgzf_deflate: on the GPU) instead of zlib here."""
    lib = hostio()
    src = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
    bounds = np.ascontiguousarray(bounds, np.int64)
    assert bounds[0] == 0 and bounds[-1] == src.size
    nb = int(lib.amp_bgzf_plan(_p(bounds), _ll(bounds.size), None, _ll(0)))
    bstart = np.empty(nb + 1, np.int64)
    assert lib.amp_bgzf_plan(_p(bounds), _ll(bounds.size), _p(bstart), _ll(nb)) == nb
    if deflater is not None:
        return deflater(src, bstart)
    out = np.empty(src.size + 64 * nb + 1024, np.uint8)
    n = lib.amp_bgzf_deflate_blocks(_p(src), _p(bstart), _ll(nb), _p(out), level, threads)
    if n < 0:
        raise RuntimeError("BGZF deflate failed")
    return out[:n].tobytes()


def bgzf_compress(data, level=6, threads=0):
    lib = hostio()
    src = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
    out = np.empty(int(lib.amp_bgzf_bound(_ll(src.size))), np.uint8)
    n = lib.amp_bgzf_deflate(_p(src), _ll(src.size), _p(out), level, threads)
    if n < 0:
        raise RuntimeError("BGZF deflate failed")
    return out[:n].tobytes()


# ------------------------------------------------------------------------------------------- containers
class Alignments:
    """Decoded input: header + ReadBatch + whatever is needed to write records back unchanged."""

    def __init__(self, fmt, header_text, refs, batch):
        self.fmt, self.header_text, self.refs, self.batch = fmt, header_text, refs, batch
        self.sam_fields = None      # SAM: list of field lists per record
        self.bam_buf = None         # BAM: decompressed byte stream (uint8) ...
        self.bam_rec_off = None     # ... and the offset of every record's block_size word

    @property
    def n(self):
        return self.batch.n


def read_alignments(path, threads=0):
    """AmpliPy.py:313-324: 'stdin' = SAM text on standard input; otherwise by extension."""
    if path.lower() == "stdin":
        return _read_sam(sys.stdin.read())
    if not os.path.isfile(path):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_NOT_FOUND, path))
    if path.lower().endswith(".sam"):
        with open(path, "r") as f:
            return _read_sam(f.read())
    if path.lower().endswith(".bam"):
        with open(path, "rb") as f:
            return _read_bam(f.read(), threads)
    raise InputError("%s: %s" % (ERROR_TEXT_INVALID_READ_EXTENSION, path))


def _read_sam(text):
    header, fields = [], []
    for line in text.splitlines():
        if not line:
            continue
        if line.startswith("@"):
            header.append(line)
        else:
            fields.append(line.split("\t"))
    n = len(fields)
    pos = np.empty(n, np.int32); flag = np.empty(n, np.uint16); tlen = np.empty(n, np.int32)
    cig_off = np.zeros(n + 1, np.int64); qual_off = np.zeros(n + 1, np.int64); seq_off = np.zeros(n + 1, np.int64)
    cig, seqs, quals = [], [], []
    for i, f in enumerate(fields):
        flag[i] = int(f[1]); pos[i] = int(f[3]) - 1; tlen[i] = int(f[8])
        ops = parse_cigar(f[5])
        cig.extend((ln << 4) | op for op, ln in ops)
        s = "" if f[9] == "*" else f[9]
        seqs.append(pack_seq(s))
        if f[10] == "*":
            q = np.full(len(s), 255, np.uint8)
        else:
            q = np.frombuffer(f[10].encode(), np.uint8) - 33
        quals.append(q)
        cig_off[i + 1] = cig_off[i] + len(ops)
        qual_off[i + 1] = qual_off[i] + len(s)
        seq_off[i + 1] = seq_off[i] + (len(s) + 1) // 2
    cat = lambda xs: np.concatenate(xs).astype(np.uint8) if xs else np.zeros(0, np.uint8)
    batch = ReadBatch(pos, flag, tlen, cig_off.astype(np.uint32), np.array(cig, np.uint32), seq_off.astype(np.uint32),
                      cat(seqs), qual_off.astype(np.uint32), cat(quals)).validate()
    refs = []
    for l in header:
        if l.startswith("@SQ"):
            d = dict(kv.split(":", 1) for kv in l.split("\t")[1:] if ":" in kv)
            refs.append((d.get("SN", "*"), int(d.get("LN", 0))))
    a = Alignments("sam", "\n".join(header) + ("\n" if header else ""), refs, batch)
    a.sam_fields = fields
    return a


def _read_bam(raw, threads=0):
    lib = hostio()
    buf = bgzf_decompress(raw, threads)
    if buf.size < 12 or bytes(buf[:4]) != b"BAM\x01":
        raise InputError("Invalid BAM file")
    try:
        l_text = int(buf[4:8].view(np.int32)[0])
        if l_text < 0 or 8 + l_text + 4 > buf.size:
            raise ValueError
        header_text = bytes(buf[8:8 + l_text]).split(b"\0", 1)[0].decode()
        p = 8 + l_text
        n_ref = int(buf[p:p + 4].view(np.int32)[0]); p += 4
        refs = []
        for _ in range(n_ref):
            l_name = int(buf[p:p + 4].view(np.int32)[0]); p += 4
            if l_name < 1 or p + l_name + 4 > buf.size:
                raise ValueError
            name = bytes(buf[p:p + l_name - 1]).decode(); p += l_name
            refs.append((name, int(buf[p:p + 4].view(np.int32)[0]))); p += 4
    except (ValueError, IndexError, UnicodeDecodeError):
        raise InputError("Invalid BAM file")
    n = lib.amp_bam_scan(_p(buf), _ll(buf.size), _ll(p), None, None, None, _ll(0))
    if n < 0:
        raise InputError("Corrupt BAM record stream")
    rec_off = np.empty(n, np.int64); ncig = np.empty(n, np.int32); lseq = np.empty(n, np.int32)
    lib.amp_bam_scan(_p(buf), _ll(buf.size), _ll(p), _p(rec_off), _p(ncig), _p(lseq), _ll(n))
    cig_off = np.zeros(n + 1, np.int64); np.cumsum(ncig, out=cig_off[1:])
    qual_off = np.zeros(n + 1, np.int64); np.cumsum(lseq, out=qual_off[1:])
    seq_off = np.zeros(n + 1, np.int64); np.cumsum((lseq.astype(np.int64) + 1) // 2, out=seq_off[1:])
    if qual_off[-1] >= 2 ** 32:
        raise InputError("BAM too large for one batch (>4 GiB of bases); split the input")
    b = ReadBatch(np.empty(n, np.int32), np.empty(n, np.uint16), np.empty(n, np.int32), cig_off.astype(np.uint32),
                  np.empty(int(cig_off[-1]), np.uint32), seq_off.astype(np.uint32), np.empty(int(seq_off[-1]), np.uint8),
                  qual_off.astype(np.uint32), np.empty(int(qual_off[-1]), np.uint8))
    lib.amp_bam_fill(_p(buf), _p(rec_off), _ll(n), _p(b.pos), _p(b.flag), _p(b.tlen), _p(b.cig_off), _p(b.cigar),
                     _p(b.seq_off), _p(b.seq), _p(b.qual_off), _p(b.qual), threads)
    a = Alignments("bam", header_text, refs, b)
    a.bam_buf, a.bam_rec_off = buf, rec_off
    return a


# ------------------------------------------------------------------------------------------- header
def header_with_pg(header_text, argv):
    """Append the @PG record the reference appends (AmpliPy.py:326-342)."""
    lines = [l for l in header_text.split("\n") if l]
    pgs = [dict(kv.split(":", 1) for kv in l.split("\t")[1:] if ":" in kv) for l in lines if l.startswith("@PG")]
    if not pgs:
        raise InputError("Input alignment header has no @PG line (AmpliPy.py:333 needs the last @PG ID)")
    n_existing = sum(1 for d in pgs if d.get("PN") == "AmpliPy")
    pg_id = "AmpliPy" if n_existing == 0 else "AmpliPy.%d" % n_existing
    lines.append("@PG\tID:%s\tPN:AmpliPy\tPP:%s\tVN:%s\tCL:%s" % (pg_id, pgs[-1].get("ID", ""), VERSION, " ".join(argv)))
    return "\n".join(lines) + "\n"


# ------------------------------------------------------------------------------------------- output
def check_output_path(path):
    """AmpliPy.py:347-356: refuse to overwrite, accept .sam / .bam / 'stdout'."""
    if path.lower() == "stdout":
        return
    if os.path.isfile(path):
        raise InputError("%s: %s" % (ERROR_TEXT_FILE_EXISTS, path))
    if not (path.lower().endswith(".sam") or path.lower().endswith(".bam")):
        raise InputError("%s: %s" % (ERROR_TEXT_INVALID_READ_EXTENSION, path))


def default_bam_level():
    """Deflate level of the BAM files written here: 6 like htslib's default; AMPLIPY_BAM_LEVEL overrides (1 = fastest)."""
    try:
        return max(0, min(9, int(os.environ.get("AMPLIPY_BAM_LEVEL", "6"))))
    except ValueError:
        return 6


def write_alignments(path, aln, header_text, trim, threads=0, level=None, deflater=None):
    """Write the reads that pass the gate (AmpliPy.py:910-911) with their new pos / CIGAR.  ``deflater``: see bgzf_compress_units
    (BAM output of BAM input only)."""
    level = default_bam_level() if level is None else level
    sel = np.flatnonzero(trim.keep).astype(np.int64)
    to_sam = path.lower() == "stdout" or path.lower().endswith(".sam")
    if to_sam:
        out = sys.stdout if path.lower() == "stdout" else open(path, "w")
        out.write(header_text)
        if aln.fmt == "sam":
            for i in sel:
                f = list(aln.sam_fields[i])
                f[3] = str(int(trim.pos[i]) + 1)
                f[5] = cigar_string(trim.cigartuples(int(i)))
                out.write("\t".join(f) + "\n")
        else:
            for i in sel:
                out.write(_bam_record_to_sam(aln, int(i), int(trim.pos[i]), trim.cigartuples(int(i))) + "\n")
        if out is not sys.stdout:
            out.close()
        return len(sel)
    # BAM output
    if aln.fmt == "bam":
        lib = hostio()
        b = aln.batch
        ooff = np.empty(len(sel) + 1, np.int64)
        lib.amp_bam_rewrite_offsets(_p(aln.bam_buf), _p(aln.bam_rec_off), _p(sel), _ll(len(sel)), _p(trim.ncig), _p(ooff))
        head = _bam_header_bytes(header_text, aln.refs)
        hb = np.frombuffer(head, np.uint8)
        size = int(ooff[-1])
        data = np.empty(hb.size + size + 8, np.uint8)               # header and records in one buffer: the stream to compress
        data[:hb.size] = hb
        lib.amp_bam_rewrite(_p(aln.bam_buf), _p(aln.bam_rec_off), _p(sel), _ll(len(sel)), _p(trim.pos), _p(trim.ncig),
                            _p(b.cig_off), _p(trim.cigar), ctypes.c_void_p(data.ctypes.data + hb.size))
        bounds = np.empty(len(sel) + 2, np.int64)                   # cut points: header end, record starts (increasing), end
        bounds[0] = 0
        bounds[1:] = ooff + hb.size
        with open(path, "wb") as f:
            f.write(bgzf_compress_units(data[:hb.size + size], bounds, level, threads, deflater))
        return len(sel)
    else:
        body = np.frombuffer(b"".join(_sam_fields_to_bam(aln, int(i), int(trim.pos[i]), trim.cigartuples(int(i))) for i in sel),
                             np.uint8)
    head = _bam_header_bytes(header_text, aln.refs)
    with open(path, "wb") as f:
        f.write(_bam_file_bytes(head, np.ascontiguousarray(body), level, threads))
    return len(sel)


def _bam_file_bytes(head, body, level, threads):
    """header + records as BGZF with htslib's layout: the header in blocks of its own, records never straddling a block"""
    lib = hostio()
    body = np.ascontiguousarray(body, np.uint8)
    n = int(lib.amp_bam_scan(_p(body), _ll(body.size), _ll(0), None, None, None, _ll(0))) if body.size else 0
    if n < 0:
        raise RuntimeError("internal error: malformed BAM records")
    rec_off = np.empty(max(n, 1), np.int64); ncig = np.empty(max(n, 1), np.int32); lseq = np.empty(max(n, 1), np.int32)
    if n:
        lib.amp_bam_scan(_p(body), _ll(body.size), _ll(0), _p(rec_off), _p(ncig), _p(lseq), _ll(n))
    hb = np.frombuffer(head, np.uint8)
    bounds = np.concatenate([[0], hb.size + rec_off[:n], [hb.size + body.size]]).astype(np.int64)
    bounds = np.unique(bounds)
    return bgzf_compress_units(np.concatenate([hb, body]), bounds, level, threads)


def _bam_header_bytes(header_text, refs):
    t = header_text.encode()
    out = [b"BAM\x01", np.int32(len(t)).tobytes(), t, np.int32(len(refs)).tobytes()]
    for name, ln in refs:
        nb = name.encode() + b"\0"
        out += [np.int32(len(nb)).tobytes(), nb, np.int32(ln).tobytes()]
    return b"".join(out)


def _reg2bin(beg, end):
    end -= 1
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return base + (beg >> shift)
    return 0


def _sam_fields_to_bam(aln, i, pos, ops):
    """One SAM record -> BAM bytes (small inputs only; the fast path is BAM -> BAM)."""
    import struct
    f = aln.sam_fields[i]
    names = [r[0] for r in aln.refs]
    rid = names.index(f[2]) if f[2] in names else -1
    nrid = rid if f[6] == "=" else (names.index(f[6]) if f[6] in names else -1)
    flag = int(f[1])
    rlen = sum(n for op, n in ops if op in (0, 2, 3, 7, 8))
    if (flag & 4) or rlen == 0:
        rlen = 1
    seq = "" if f[9] == "*" else f[9]
    qual = bytes([255] * len(seq)) if f[10] == "*" else bytes(c - 33 for c in f[10].encode())
    name = f[0].encode() + b"\0"
    tags = b"".join(_sam_tag_to_bam(t) for t in f[11:])
    core = struct.pack("<iiBBHHHiiii", rid, pos, len(name), int(f[4]), _reg2bin(pos, pos + rlen), len(ops), flag, len(seq),
                       nrid, int(f[7]) - 1, int(f[8]))
    body = core + name + b"".join(struct.pack("<I", (n << 4) | op) for op, n in ops) + pack_seq(seq).tobytes() + qual + tags
    return struct.pack("<I", len(body)) + body


def _sam_tag_to_bam(t):
    import struct
    tag, typ, val = t.split(":", 2)
    k = tag.encode()
    if typ == "A":
        return k + b"A" + val.encode()
    if typ == "i":
        v = int(val)
        for code, fmt, lo, hi in (("C", "<B", 0, 255), ("c", "<b", -128, 127), ("S", "<H", 0, 65535), ("s", "<h", -32768, 32767),
                                  ("I", "<I", 0, 2 ** 32 - 1), ("i", "<i", -2 ** 31, 2 ** 31 - 1)):
            if lo <= v <= hi:
                return k + code.encode() + struct.pack(fmt, v)
    if typ == "f":
        return k + b"f" + struct.pack("<f", float(val))
    if typ == "Z":
        return k + b"Z" + val.encode() + b"\0"
    if typ == "H":
        return k + b"H" + val.encode() + b"\0"
    if typ == "B":
        parts = val.split(",")
        sub = parts[0]
        fmt = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I", "f": "<f"}[sub]
        conv = float if sub == "f" else int
        return k + b"B" + sub.encode() + struct.pack("<i", len(parts) - 1) + b"".join(struct.pack(fmt, conv(x)) for x in parts[1:])
    raise InputError("Unsupported SAM tag type: %s" % t)


def _bam_record_to_sam(aln, i, pos, ops):
    import struct
    buf = aln.bam_buf
    o = int(aln.bam_rec_off[i])
    bs = int(buf[o:o + 4].view(np.uint32)[0])
    r = bytes(buf[o + 4:o + 4 + bs])
    rid, _pos, lname, mapq, _bin, ncig, flag, lseq, nrid, npos, tlen = struct.unpack("<iiBBHHHiiii", r[:32])
    name = r[32:32 + lname - 1].decode()
    p = 32 + lname + 4 * ncig
    rec = aln.batch.record(i)
    p += (lseq + 1) // 2
    q = r[p:p + lseq]; p += lseq
    qual = "*" if (lseq == 0 or q[0] == 255) else "".join(chr(c + 33) for c in q)
    names = [x[0] for x in aln.refs]
    rname = names[rid] if rid >= 0 else "*"
    rnext = "*" if nrid < 0 else ("=" if nrid == rid else names[nrid])
    fields = [name, str(flag), rname, str(pos + 1), str(mapq), cigar_string(ops), rnext, str(npos + 1), str(tlen),
              rec[4] if lseq else "*", qual] + _bam_tags_to_sam(r[p:])
    return "\t".join(fields)


def _bam_tags_to_sam(b):
    import struct
    out = []
    p = 0
    sizes = {"c": ("<b", 1), "C": ("<B", 1), "s": ("<h", 2), "S": ("<H", 2), "i": ("<i", 4), "I": ("<I", 4), "f": ("<f", 4)}
    while p + 3 <= len(b):
        tag = b[p:p + 2].decode(); t = chr(b[p + 2]); p += 3
        if t == "A":
            out.append("%s:A:%s" % (tag, chr(b[p]))); p += 1
        elif t in sizes:
            fmt, n = sizes[t]
            v = struct.unpack(fmt, b[p:p + n])[0]; p += n
            out.append("%s:%s:%s" % (tag, "f" if t == "f" else "i", ("%g" % v) if t == "f" else v))
        elif t in "ZH":
            e = b.index(b"\0", p)
            out.append("%s:%s:%s" % (tag, t, b[p:e].decode())); p = e + 1
        elif t == "B":
            sub = chr(b[p]); cnt = struct.unpack("<i", b[p + 1:p + 5])[0]; p += 5
            fmt, n = sizes[sub]
            vals = [struct.unpack(fmt, b[p + k * n:p + (k + 1) * n])[0] for k in range(cnt)]; p += cnt * n
            out.append("%s:B:%s,%s" % (tag, sub, ",".join(("%g" % v) if sub == "f" else str(v) for v in vals)))
        else:
            break
    return out


def write_bam(path, header_text, refs, batch, names=None, mapq=60, threads=0, level=1, refid=None):
    """Serialise a ReadBatch as a BAM file (synthetic inputs for tests / benchmarks; read names r<i>).  ``refid``: the refID of
    every read (also its mate's, for paired reads); default 0, and -1 for unmapped reads."""
    lib = hostio()
    b = batch
    nblob = noff = None
    if names is not None:
        enc = [str(x).encode() + b"\0" for x in names]
        assert len(enc) == b.n and all(len(e) <= 255 for e in enc)
        noff = np.zeros(b.n + 1, np.int64)
        np.cumsum([len(e) for e in enc], out=noff[1:])
        nblob = np.frombuffer(b"".join(enc) + b"\0", np.uint8)
    args = (_ll(b.n), _p(b.pos), _p(b.flag), _p(b.tlen), _p(b.cig_off), _p(b.cigar), _p(b.seq_off), _p(b.seq), _p(b.qual_off),
            _p(b.qual), int(mapq), _p(nblob), _p(noff))
    size = int(lib.amp_bam_serialize(*args, None, None))
    body = np.empty(size + 8, np.uint8)
    rec_off = np.empty(b.n + 1, np.int64)
    lib.amp_bam_serialize(*args, _p(body), _p(rec_off))
    if refid is not None:
        rid = np.ascontiguousarray(refid, np.int32)
        assert rid.shape == (b.n,)
        at = rec_off[:-1, None] + np.arange(4)
        body[at + 4] = rid.view(np.uint8).reshape(-1, 4)
        paired = np.flatnonzero(b.flag & 1)
        body[at[paired] + 24] = rid[paired].view(np.uint8).reshape(-1, 4)
    with open(path, "wb") as f:
        f.write(_bam_file_bytes(_bam_header_bytes(header_text, refs), body[:size], level, threads))
