"""ctypes binding of libamplipy_b200.so (include/amplipy_b200.h) -- the host-side mirror of the
reference's per-read / per-position functions, operating on whole batches:

    reference (AmpliPy.py)                      here
    ------------------------------------------  ---------------------------------------------
    find_overlapping_primers (174-209)          primers.find_overlapping_primers -> Engine(...)
    trim_read (426-687) + write gate (910)      Engine.process(batch, trim=True)   -> TrimResult
    update_base_counts (690-753)                Engine.process(batch, pileup=True) -> counts()/insertions()
    alleles_from_counts + call loop (756-951)   Engine.call(ref_seq, ...)          -> CallResult

There is no CPU fallback: if the CUDA library is missing or no GPU is present, this module raises.
PyTorch is used only for device buffers / streams (``upload`` + ``process_device``).
"""
import ctypes
import os

import numpy as np

from .batch import ReadBatch
from .calling import CallResult, Insertions
from .ivar import Annotation, Deletions, IvarResult, QStats

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AMP_LIB_OVERRIDE") or os.path.join(_HERE, "csrc", "libamplipy_b200.so")   # override: tuning experiments only

MODE_TRIM, MODE_PILEUP, MODE_QSTATS = 1, 2, 4
F_TRIM_START, F_TRIM_END, F_TRIM_QUAL, F_KEEP, F_SKIPPED, F_ERROR = 1, 2, 4, 8, 16, 32
DEVERR_NAMES = {1: "read outside the reference (IndexError in AmpliPy.py:450-451)",
                2: "aligned base not in ACGTN (KeyError in AmpliPy.py:753)",
                4: "insertion runs to the end of the alignment (IndexError in AmpliPy.py:734)",
                8: "CIGAR consumes more query than l_seq / unsupported op",
                16: "insertion hash table full (raise ins_slots)",
                32: "insertion string arena full (raise ins_arena_bytes)",
                64: "strand / quality pass met an insertion allele the pileup did not add",
                128: "anchored deletion table full (raise the slots of enable_dels)"}

EXPORTED_SYMBOLS = [
    "amp_last_error", "amp_abi_version", "amp_create", "amp_destroy", "amp_reset", "amp_error_flags", "amp_lpad",
    "amp_sm_count", "amp_process_device", "amp_process_host", "amp_last_launches", "amp_counts_device",
    "amp_bind_counts", "amp_counts_host", "amp_ins_count", "amp_ins_export", "amp_ins_merge", "amp_call",
    "amp_host_alloc", "amp_host_free", "amp_reset_async", "amp_set_reference", "amp_call_device",
    "amp_nccl_unique_id", "amp_nccl_comm_init", "amp_nccl_comm_destroy", "amp_nccl_allgather", "amp_allreduce_counts",
    "amp_ins_slot_bytes", "amp_ins_pack_device", "amp_ins_merge_packed", "amp_reserve", "amp_counts_copy_device",
    "amp_bam_decode_host", "amp_process_decoded", "amp_decoded_copy_host", "amp_counts_upload", "amp_bgzf_deflate_host", "amp_decoded_write_bam",
    "amp_set_scheme", "amp_get_scheme", "amp_set_sample_reference", "amp_qstats_enable", "amp_qstats_host", "amp_call_ivar",
    "amp_call_ivar_device", "amp_contig_plan_decoded", "amp_contig_plan_device", "amp_process_contigs", "amp_set_features",
    "amp_annotate", "amp_annot_host", "amp_allreduce_qstats", "amp_ins_slot_bytes_qstats", "amp_ins_pack_qstats_device",
    "amp_ins_merge_packed_qstats", "amp_dels_enable", "amp_dels_count", "amp_dels_export", "amp_dels_merge", "amp_call_ivar_dels",
    "amp_dels_slot_bytes", "amp_dels_pack_device", "amp_dels_merge_packed"]


class AmpConfig(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int32), ("ref_len", ctypes.c_int32), ("n_samples", ctypes.c_int32),
                ("min_quality", ctypes.c_int32), ("sliding_window", ctypes.c_int32), ("min_length", ctypes.c_int32),
                ("include_no_primer", ctypes.c_int32), ("ins_slots", ctypes.c_int64), ("ins_arena_bytes", ctypes.c_int64)]


class AmpBatch(ctypes.Structure):
    _fields_ = [("first", ctypes.c_int64), ("n_reads", ctypes.c_int64), ("pos", ctypes.c_void_p),
                ("flag", ctypes.c_void_p), ("tlen", ctypes.c_void_p), ("cig_off", ctypes.c_void_p),
                ("cigar", ctypes.c_void_p), ("seq_off", ctypes.c_void_p), ("seq", ctypes.c_void_p),
                ("qual_off", ctypes.c_void_p), ("qual", ctypes.c_void_p)]


class AmpTrimOut(ctypes.Structure):
    _fields_ = [("pos", ctypes.c_void_p), ("ncig", ctypes.c_void_p), ("flags", ctypes.c_void_p),
                ("cigar", ctypes.c_void_p)]


class AmpBamInfo(ctypes.Structure):
    _fields_ = [("n_reads", ctypes.c_int64), ("sum_cigar_ops", ctypes.c_int64), ("sum_seq_bytes", ctypes.c_int64),
                ("sum_qual_bytes", ctypes.c_int64), ("raw_bytes", ctypes.c_int64)]


class AmpBatchOut(ctypes.Structure):
    _fields_ = [("pos", ctypes.c_void_p), ("flag", ctypes.c_void_p), ("tlen", ctypes.c_void_p), ("cig_off", ctypes.c_void_p),
                ("cigar", ctypes.c_void_p), ("seq_off", ctypes.c_void_p), ("seq", ctypes.c_void_p), ("qual_off", ctypes.c_void_p),
                ("qual", ctypes.c_void_p)]


class AmpContigPlan(ctypes.Structure):
    _fields_ = [("n_reads", ctypes.c_int64), ("n_no_contig", ctypes.c_int64), ("grouped", ctypes.c_int32), ("errors", ctypes.c_uint32),
                ("contig_reads", ctypes.c_void_p), ("contig_first", ctypes.c_void_p), ("contig_cigar_ops", ctypes.c_void_p),
                ("contig_qual_bytes", ctypes.c_void_p), ("ref_reads", ctypes.c_void_p)]


CONTIG_E_NOFLAG4, CONTIG_E_UNKNOWN, CONTIG_E_BADID = 1, 2, 4


class ContigPlan:
    """What amp_contig_plan_* found in a batch: per contig (= sample) its reads, first read, CIGAR ops and quality bytes; the
    reads without a contig; whether every contig's reads are contiguous; error bits (CONTIG_E_*) and, for a decoded BAM, the
    reads on each header sequence that is not in the FASTA."""

    def __init__(self, n_samples, n_refs=0):
        self.reads, self.first = np.zeros(n_samples, np.int64), np.zeros(n_samples, np.int64)
        self.cigar_ops, self.qual_bytes = np.zeros(n_samples, np.int64), np.zeros(n_samples, np.int64)
        self.ref_reads = np.zeros(max(n_refs, 1), np.int64)[:n_refs]
        self.c = AmpContigPlan(0, 0, 0, 0, _ptr(self.reads), _ptr(self.first), _ptr(self.cigar_ops), _ptr(self.qual_bytes),
                               _ptr(self.ref_reads) if n_refs else None)

    n_reads = property(lambda self: int(self.c.n_reads))
    n_no_contig = property(lambda self: int(self.c.n_no_contig))
    grouped = property(lambda self: bool(self.c.grouped))
    errors = property(lambda self: int(self.c.errors))


class AmpCallParams(ctypes.Structure):
    _fields_ = [("min_depth_consensus", ctypes.c_int32), ("min_freq_consensus", ctypes.c_double),
                ("min_depth_variants", ctypes.c_int32), ("min_freq_variants", ctypes.c_double)]


class AmpIvarParams(ctypes.Structure):
    _fields_ = [("min_depth", ctypes.c_int32), ("min_freq", ctypes.c_double), ("iupac_threshold", ctypes.c_double)]


class AmpCallOut(ctypes.Structure):
    _fields_ = [("depth", ctypes.c_void_p), ("top_id", ctypes.c_void_p), ("top_count", ctypes.c_void_p),
                ("pos_flags", ctypes.c_void_p), ("ref_count", ctypes.c_void_p), ("fixed_freq", ctypes.c_void_p),
                ("fixed_rank", ctypes.c_void_p), ("alt_mask", ctypes.c_void_p)]


_lib = None


def load_library():
    """dlopen the C-ABI library; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError("amplipy_b200: %s is missing -- build it with `python -m amplipy_b200.build` "
                               "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        lib.amp_last_error.restype = ctypes.c_char_p
        lib.amp_ins_slot_bytes.restype = ctypes.c_int64
        lib.amp_ins_slot_bytes_qstats.restype = ctypes.c_int64
        if hasattr(lib, "amp_dels_slot_bytes"):       # A/B runs may load a library from before the deletion table
            lib.amp_dels_slot_bytes.restype = ctypes.c_int64
        for name in EXPORTED_SYMBOLS:
            try:
                getattr(lib, name)   # AttributeError if the build is stale
            except AttributeError:
                if not (os.environ.get("AMP_LIB_OVERRIDE") and os.environ.get("AMP_LIB_ALLOW_MISSING")):   # A/B runs against older kernels
                    raise
        _lib = lib
    return _lib


class AmpError(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        raise AmpError("%s failed (%d): %s" % (what, rc, load_library().amp_last_error().decode()))


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


class ContigError(AmpError):
    """amp_contig_plan_* flagged reads without a valid contig (``plan.errors``); nothing was processed."""

    def __init__(self, plan):
        super().__init__("contig plan error bits 0x%x" % plan.errors)
        self.plan = plan


class TrimResult:
    """Per-read outputs of the trim kernel (row i of ``cigar`` starts at cig_off[i] + 3*i)."""

    def __init__(self, batch, pos, ncig, flags, cigar):
        self.batch, self.pos, self.ncig, self.flags, self.cigar = batch, pos, ncig, flags, cigar

    def cigartuples(self, i):
        a = int(self.batch.cig_off[i]) + 3 * i
        return [(int(c & 15), int(c >> 4)) for c in self.cigar[a:a + int(self.ncig[i])]]

    @property
    def keep(self):
        return (self.flags & F_KEEP) != 0

    def trimmed_batch(self, only_kept=True):
        """The trimmed reads as a new ReadBatch (what the reference writes with out_aln.write, 911)."""
        b = self.batch
        sel = np.flatnonzero(self.keep) if only_kept else np.flatnonzero((self.flags & (F_SKIPPED | F_ERROR)) == 0)
        ncig = self.ncig[sel].astype(np.int64)
        new_off = np.zeros(len(sel) + 1, np.int64)
        np.cumsum(ncig, out=new_off[1:])
        row0 = b.cig_off[:-1].astype(np.int64)[sel] + 3 * sel
        idx = np.repeat(row0 - new_off[:-1], ncig) + np.arange(int(new_off[-1]), dtype=np.int64)
        cig = self.cigar[idx]

        def gather(off, data):
            off = off.astype(np.int64)
            ln = np.diff(off)[sel]
            no = np.zeros(len(sel) + 1, np.int64)
            np.cumsum(ln, out=no[1:])
            ii = np.repeat(off[:-1][sel] - no[:-1], ln) + np.arange(int(no[-1]), dtype=np.int64)
            return no.astype(np.uint32), np.ascontiguousarray(data[ii])
        so, s = gather(b.seq_off, b.seq)
        qo, q = gather(b.qual_off, b.qual)
        return ReadBatch(np.ascontiguousarray(self.pos[sel]), np.ascontiguousarray(b.flag[sel]),
                         np.ascontiguousarray(b.tlen[sel]), new_off.astype(np.uint32), np.ascontiguousarray(cig),
                         so, s, qo, q), sel


class Engine:
    def __init__(self, ref_len, primer_tables=None, max_primer_len=0, min_quality=20, sliding_window_width=4,
                 min_length=30, include_no_primer=False, n_samples=1, device=0, ins_slots=0, ins_arena_bytes=0):
        """primer_tables = (min_primer_start, max_primer_end) int32[L] with -1 for uncovered positions
        (``primers.find_overlapping_primers``); None for pileup/calling-only use."""
        self.lib = load_library()
        self.L = int(ref_len)
        self.n_samples = int(n_samples)
        cfg = AmpConfig(device, self.L, n_samples, min_quality, sliding_window_width, min_length,
                        1 if include_no_primer else 0, ins_slots, ins_arena_bytes)
        self._ctx = ctypes.c_void_p()
        mn = mx = None
        if primer_tables is not None:
            mn = np.ascontiguousarray(primer_tables[0], np.int32)
            mx = np.ascontiguousarray(primer_tables[1], np.int32)
            assert mn.shape == (self.L,) and mx.shape == (self.L,)
        _check(self.lib.amp_create(ctypes.byref(cfg), _ptr(mn), _ptr(mx), ctypes.c_int32(int(max_primer_len)),
                                   ctypes.byref(self._ctx)), "amp_create")
        self.has_primers = primer_tables is not None
        self.lpad = int(self.lib.amp_lpad(self._ctx))
        self.device = device
        self.launches = 0
        self._qstats = False
        self._dels = False

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.amp_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _check(self.lib.amp_reset(self._ctx), "amp_reset")

    def reset_async(self, stream=None):
        _check(self.lib.amp_reset_async(self._ctx, ctypes.c_void_p(stream) if stream else None), "amp_reset_async")
        self.launches += 2 if self._dels else 1      # amp_reset_kernel (+ amp_dels_reset_kernel)

    def set_reference(self, ref_seq):
        ref = ref_seq.encode("latin-1") if isinstance(ref_seq, str) else bytes(ref_seq)
        assert len(ref) == self.L
        _check(self.lib.amp_set_reference(self._ctx, ctypes.c_char_p(ref)), "amp_set_reference")

    # ---------------------------------------------------------------- heterogeneous plates: a scheme / reference per sample
    def set_scheme(self, sample, primers, offset=0, ref_len=None):
        """Primer scheme of one sample: [(start, end)] sorted as load_primers returns them; the two per-position tables are
        built on the device (find_overlapping_primers, AmpliPy.py:174-209)."""
        st = np.ascontiguousarray([p[0] for p in primers], np.int32)
        en = np.ascontiguousarray([p[1] for p in primers], np.int32)
        _check(self.lib.amp_set_scheme(self._ctx, int(sample), int(self.L if ref_len is None else ref_len), _ptr(st), _ptr(en),
                                       int(st.size), int(offset)), "amp_set_scheme")
        self.has_primers = True

    def get_scheme(self, sample, ref_len=None):
        n = int(self.L if ref_len is None else ref_len)
        mn, mx = np.empty(n, np.int32), np.empty(n, np.int32)
        mpl = ctypes.c_int32(0)
        _check(self.lib.amp_get_scheme(self._ctx, int(sample), _ptr(mn), _ptr(mx), ctypes.byref(mpl)), "amp_get_scheme")
        return mn, mx, int(mpl.value)

    def set_sample_reference(self, sample, ref_seq):
        ref = ref_seq.encode("latin-1") if isinstance(ref_seq, str) else bytes(ref_seq)
        _check(self.lib.amp_set_sample_reference(self._ctx, int(sample), ctypes.c_char_p(ref), len(ref)), "amp_set_sample_reference")

    def call_device(self, min_depth_consensus=10, min_freq_consensus=0.0, min_depth_variants=1, min_freq_variants=0.03,
                    stream=None):
        cp = AmpCallParams(int(min_depth_consensus), float(min_freq_consensus), int(min_depth_variants),
                           float(min_freq_variants))
        _check(self.lib.amp_call_device(self._ctx, ctypes.byref(cp), ctypes.c_void_p(stream) if stream else None),
               "amp_call_device")
        self.launches += int(self.lib.amp_last_launches(self._ctx))

    def sm_count(self):
        return int(self.lib.amp_sm_count(self._ctx))

    def error_flags(self):
        f = ctypes.c_uint32(0)
        _check(self.lib.amp_error_flags(self._ctx, ctypes.byref(f)), "amp_error_flags")
        return int(f.value)

    def raise_on_device_errors(self):
        f = self.error_flags()
        if f:
            raise AmpError("; ".join(v for k, v in DEVERR_NAMES.items() if f & k))

    # ---------------------------------------------------------------- host-buffer path (e2e)
    @staticmethod
    def alloc_trim_out(batch):
        # zero-initialised: process(first, n) fills only [first, first + n); flags == 0 means "not kept" for the other reads
        n = batch.n
        return (np.zeros(n, np.int32), np.zeros(n, np.uint16), np.zeros(n, np.uint8),
                np.zeros(int(batch.cig_off[-1]) + 3 * n, np.uint32))

    def process(self, batch, trim=True, pileup=True, sample=0, out=None, first=0, n=None, qstats=False):
        """H2D + fused kernel + D2H through amp_process_host.  Returns TrimResult when trim=True.  ``qstats=True``: the
        strand / quality pass runs on the same reads (enable_qstats first)."""
        mode = (MODE_TRIM if trim else 0) | (MODE_PILEUP if pileup else 0) | (MODE_QSTATS if qstats else 0)
        n = batch.n - first if n is None else n
        hb = AmpBatch(first, n, _ptr(batch.pos), _ptr(batch.flag), _ptr(batch.tlen), _ptr(batch.cig_off),
                      _ptr(batch.cigar), _ptr(batch.seq_off), _ptr(batch.seq), _ptr(batch.qual_off), _ptr(batch.qual))
        to = None
        if trim:
            if out is None:
                out = self.alloc_trim_out(batch)
            to = AmpTrimOut(_ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]))
        _check(self.lib.amp_process_host(self._ctx, ctypes.byref(hb), mode, sample, ctypes.byref(to) if to else None),
               "amp_process_host")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return TrimResult(batch, *out) if trim else None

    def host_copy_bytes(self, batch, trim=True, pileup=True, call=True):
        """(host->device, device->host) bytes one `process` (+ `call`) of this batch moves over PCIe, counted from the
        arrays the C ABI copies: inputs = the batch's nine arrays, outputs = the trim rows + the calling arrays."""
        n, sc = batch.n, int(batch.cig_off[-1])
        h2d = n * (4 + 2 + 4) + 3 * 4 * (n + 1) + 4 * sc + int(batch.qual.size) + (int(batch.seq.size) if pileup else 0)
        d2h = (n * (4 + 2 + 1) + 4 * (sc + 3 * n)) if trim else 0
        if call:
            d2h += self.n_samples * self.L * (4 + 4 + 4 + 1 + 4 + 48 + 24 + 1)
        return h2d, d2h

    # ---------------------------------------------------------------- device-resident path (kernel-only)
    def upload(self, batch, trim_out=True):
        """Copy a batch into HBM as torch tensors (device buffers only; no torch ops on the data)."""
        import torch
        dev = torch.device("cuda", self.device)

        def up(a):
            return torch.from_numpy(a).to(dev, non_blocking=False)

        def up_rows(a):   # seq / qual: readable up to the next 16-byte boundary past the end (include/amplipy_b200.h)
            t = torch.zeros(a.size + 16, dtype=torch.uint8, device=dev)
            if a.size:
                t[:a.size].copy_(torch.from_numpy(a))
            return t
        d = {"n": batch.n, "sum_cig": int(batch.cig_off[-1]), "sum_qual": int(batch.qual_off[-1])}
        # views of narrower dtypes that torch lacks are uploaded as raw bytes
        d["pos"] = up(batch.pos)
        d["flag"] = up(batch.flag.view(np.int16))
        d["tlen"] = up(batch.tlen)
        d["cig_off"] = up(batch.cig_off.view(np.int32))
        d["cigar"] = up(batch.cigar.view(np.int32)) if batch.cigar.size else torch.zeros(1, dtype=torch.int32, device=dev)
        d["seq_off"] = up(batch.seq_off.view(np.int32))
        d["seq"] = up_rows(batch.seq)
        d["qual_off"] = up(batch.qual_off.view(np.int32))
        d["qual"] = up_rows(batch.qual)
        if trim_out:
            d["o_pos"] = torch.empty(batch.n, dtype=torch.int32, device=dev)
            d["o_ncig"] = torch.empty(batch.n, dtype=torch.int16, device=dev)
            d["o_flags"] = torch.empty(batch.n, dtype=torch.uint8, device=dev)
            d["o_cigar"] = torch.empty(d["sum_cig"] + 3 * batch.n + 1, dtype=torch.int32, device=dev)
        return d

    def process_device(self, d, trim=True, pileup=True, sample=0, stream=None, first=0, n=None, sum_cig=None,
                       sum_qual=None, qstats=False):
        """Launch the fused kernel on a batch already resident in HBM (asynchronous on ``stream``); ``qstats=True``: and the
        strand / quality pass after it."""
        mode = (MODE_TRIM if trim else 0) | (MODE_PILEUP if pileup else 0) | (MODE_QSTATS if qstats else 0)
        n = d["n"] - first if n is None else n
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        db = AmpBatch(first, n, p(d["pos"]), p(d["flag"]), p(d["tlen"]), p(d["cig_off"]), p(d["cigar"]),
                      p(d["seq_off"]), p(d["seq"]), p(d["qual_off"]), p(d["qual"]))
        to = AmpTrimOut(p(d["o_pos"]), p(d["o_ncig"]), p(d["o_flags"]), p(d["o_cigar"])) if trim else None
        _check(self.lib.amp_process_device(self._ctx, ctypes.byref(db),
                                           ctypes.c_int64(d["sum_cig"] if sum_cig is None else sum_cig),
                                           ctypes.c_int64(d["sum_qual"] if sum_qual is None else sum_qual), mode, sample,
                                           ctypes.byref(to) if to else None,
                                           ctypes.c_void_p(stream) if stream else None), "amp_process_device")
        self.launches += int(self.lib.amp_last_launches(self._ctx))

    def download_trim(self, batch, d):
        return TrimResult(batch, d["o_pos"].cpu().numpy(), d["o_ncig"].cpu().numpy().view(np.uint16),
                          d["o_flags"].cpu().numpy(), d["o_cigar"].cpu().numpy().view(np.uint32)[:-1])

    # ---------------------------------------------------------------- results
    def counts(self, sample=0):
        out = np.empty((6, self.L), np.int32)
        _check(self.lib.amp_counts_host(self._ctx, sample, _ptr(out)), "amp_counts_host")
        return out

    def upload_counts(self, counts, sample=0):
        """Replace count matrix ``sample`` by the host array counts[6, L] (A C G T N '-')."""
        a = np.ascontiguousarray(counts, np.int32)
        assert a.shape == (6, self.L)
        _check(self.lib.amp_counts_upload(self._ctx, sample, _ptr(a)), "amp_counts_upload")

    def counts_device_ptr(self):
        p = ctypes.c_void_p()
        _check(self.lib.amp_counts_device(self._ctx, ctypes.byref(p)), "amp_counts_device")
        return p.value

    def counts_tensor(self):
        """The int32 device tensor [n_samples, 6, lpad] the kernels accumulate into (allocated through torch on first use
        so that torch.distributed can all-reduce it in place; what has been accumulated so far is carried over with a
        device-to-device copy).  The NCCL path of dist.py does not need it: amp_allreduce_counts works on the
        context's own matrix."""
        if getattr(self, "_bound", None) is None:
            import torch
            dev = torch.device("cuda", self.device)
            t = torch.empty((self.n_samples, 6, self.lpad), dtype=torch.int32, device=dev)
            _check(self.lib.amp_counts_copy_device(self._ctx, ctypes.c_void_p(t.data_ptr()), None), "amp_counts_copy_device")
            torch.cuda.synchronize(dev)
            self.bind_counts(t)
        return self._bound

    def bind_counts(self, tensor):
        """Use a caller-owned int32 device tensor [n_samples, 6, lpad] (e.g. to all-reduce it with NCCL)."""
        assert tensor.is_cuda and tensor.is_contiguous() and tensor.numel() == self.n_samples * 6 * self.lpad
        self._bound = tensor
        _check(self.lib.amp_bind_counts(self._ctx, ctypes.c_void_p(tensor.data_ptr())), "amp_bind_counts")

    def insertions(self):
        n = ctypes.c_int64(0)
        nch = ctypes.c_int64(0)
        _check(self.lib.amp_ins_count(self._ctx, ctypes.byref(n), ctypes.byref(nch)), "amp_ins_count")
        k = int(n.value)
        sample = np.empty(k, np.int32)
        pos = np.empty(k, np.int32)
        count = np.empty(k, np.int32)
        off = np.zeros(k + 1, np.int64)
        chars = np.empty(max(int(nch.value), 1), np.uint8)
        _check(self.lib.amp_ins_export(self._ctx, _ptr(sample), _ptr(pos), _ptr(count), _ptr(off), _ptr(chars)),
               "amp_ins_export")
        raw = chars.tobytes()
        strs = [raw[int(off[j]):int(off[j + 1])].decode("latin-1") for j in range(k)]
        ins = Insertions(sample, pos, count, strs)
        ins.str_off, ins.chars = off, chars[:int(off[-1])]
        return ins

    def merge_insertions(self, sample, pos, count, str_off, chars):
        sample = np.ascontiguousarray(sample, np.int32)
        pos = np.ascontiguousarray(pos, np.int32)
        count = np.ascontiguousarray(count, np.int32)
        str_off = np.ascontiguousarray(str_off, np.int64)
        chars = np.ascontiguousarray(chars, np.uint8) if len(chars) else np.zeros(1, np.uint8)
        _check(self.lib.amp_ins_merge(self._ctx, ctypes.c_int64(len(pos)), _ptr(sample), _ptr(pos), _ptr(count),
                                      _ptr(str_off), _ptr(chars)), "amp_ins_merge")

    # ---------------------------------------------------------------- BAM decoded on the device
    def decode_bam(self, raw, layout):
        """H2D of the compressed file as it is + inflate / record scan / scatter on the device (amp_bam_decode_host).
        ``raw``: the file's bytes (bytes or a uint8 array; page-locked memory makes the copy asynchronous), ``layout``:
        alnio.bam_layout(raw).  Returns the batch's totals; the batch itself stays in HBM for process_decoded()."""
        src = raw if isinstance(raw, np.ndarray) else np.frombuffer(raw, np.uint8)
        in_off = np.ascontiguousarray(layout["in_off"], np.int64)
        out_len = np.ascontiguousarray(layout["out_len"], np.uint32)
        info = AmpBamInfo()
        _check(self.lib.amp_bam_decode_host(self._ctx, _ptr(src), ctypes.c_int64(src.size), _ptr(in_off), _ptr(out_len),
                                            ctypes.c_int64(in_off.size), ctypes.c_int64(int(layout["body_off"])), ctypes.byref(info)),
               "amp_bam_decode_host")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        self._decoded = {"n": int(info.n_reads), "sum_cig": int(info.sum_cigar_ops), "sum_seq": int(info.sum_seq_bytes),
                         "sum_qual": int(info.sum_qual_bytes), "raw_bytes": int(info.raw_bytes)}
        return dict(self._decoded)

    def alloc_decoded_trim_out(self):
        n, sc = self._decoded["n"], self._decoded["sum_cig"]
        return (np.zeros(n, np.int32), np.zeros(n, np.uint16), np.zeros(n, np.uint8), np.zeros(sc + 3 * n, np.uint32))

    def process_decoded(self, trim=True, pileup=True, sample=0, out=None, download=True, qstats=False):
        """Fused kernel on the batch decode_bam left in HBM; trim outputs copied to ``out`` (alloc_decoded_trim_out), or left on the
        device only (``download=False``: decoded_write_bam is their consumer).  ``qstats=True``: the strand / quality pass too."""
        mode = (MODE_TRIM if trim else 0) | (MODE_PILEUP if pileup else 0) | (MODE_QSTATS if qstats else 0)
        to = None
        if trim and download:
            if out is None:
                out = self.alloc_decoded_trim_out()
            to = AmpTrimOut(_ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]))
        _check(self.lib.amp_process_decoded(self._ctx, mode, sample, ctypes.byref(to) if to else None), "amp_process_decoded")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return out

    # ---------------------------------------------------------------- multi-contig references (DESIGN.md 3.8): contig k = sample k
    def contig_plan_decoded(self, ref_to_sample):
        """Contig of every read of the batch decode_bam left in HBM: its BAM refID through ``ref_to_sample`` (one entry per header
        sequence: the sample, -1 = no contig, -2 = not in the FASTA).  Returns a ContigPlan."""
        m = np.ascontiguousarray(ref_to_sample, np.int32)
        plan = ContigPlan(self.n_samples, m.size)
        _check(self.lib.amp_contig_plan_decoded(self._ctx, _ptr(m) if m.size else None, int(m.size), ctypes.byref(plan.c)),
               "amp_contig_plan_decoded")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        self.contig_plan = plan
        return plan

    def process_decoded_contigs(self, trim=True, pileup=True, qstats=False, download=True, out=None):
        """The fused kernel once per contig over the planned decoded batch (contig_plan_decoded first): trim outputs in input order,
        copied to ``out`` (alloc_decoded_trim_out) unless ``download=False`` (decoded_write_bam reads them on the device)."""
        mode = (MODE_TRIM if trim else 0) | (MODE_PILEUP if pileup else 0) | (MODE_QSTATS if qstats else 0)
        to = None
        if trim and download:
            if out is None:
                out = self.alloc_decoded_trim_out()
            to = AmpTrimOut(_ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]))
        _check(self.lib.amp_process_contigs(self._ctx, mode, None, ctypes.byref(to) if to else None), "amp_process_contigs")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return out

    def process_contigs(self, batch, sample_of_read, trim=True, pileup=True, qstats=False):
        """A host batch whose read i belongs to sample_of_read[i] (-1: no contig; such a read must carry flag 4): uploaded, planned
        (self.contig_plan) and processed by the same device routine as the decoded path.  Returns TrimResult when trim=True; raises
        ContigError when the plan has error bits."""
        import torch
        sid = np.ascontiguousarray(sample_of_read, np.int32)
        assert sid.shape == (batch.n,)
        d = self.upload(batch, trim_out=trim)
        dsid = torch.from_numpy(sid).to(torch.device("cuda", self.device)) if batch.n else torch.zeros(1, dtype=torch.int32,
                                                                                                    device=torch.device("cuda", self.device))
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        db = AmpBatch(0, batch.n, p(d["pos"]), p(d["flag"]), p(d["tlen"]), p(d["cig_off"]), p(d["cigar"]), p(d["seq_off"]), p(d["seq"]),
                      p(d["qual_off"]), p(d["qual"]))
        plan = ContigPlan(self.n_samples)
        _check(self.lib.amp_contig_plan_device(self._ctx, ctypes.byref(db), p(dsid), ctypes.byref(plan.c)), "amp_contig_plan_device")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        self.contig_plan = plan
        if plan.errors:
            raise ContigError(plan)
        mode = (MODE_TRIM if trim else 0) | (MODE_PILEUP if pileup else 0) | (MODE_QSTATS if qstats else 0)
        dto = hto = out = None
        if trim:
            out = self.alloc_trim_out(batch)
            dto = AmpTrimOut(p(d["o_pos"]), p(d["o_ncig"]), p(d["o_flags"]), p(d["o_cigar"]))
            hto = AmpTrimOut(_ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]))
        _check(self.lib.amp_process_contigs(self._ctx, mode, ctypes.byref(dto) if dto else None, ctypes.byref(hto) if hto else None),
               "amp_process_contigs")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return TrimResult(batch, *out) if trim else None

    def decoded_batch(self):
        """The decoded batch copied back to the host as a ReadBatch, plus the offset of every record in the inflated stream."""
        d = self._decoded
        n = d["n"]
        b = ReadBatch(np.empty(n, np.int32), np.empty(n, np.uint16), np.empty(n, np.int32), np.empty(n + 1, np.uint32),
                      np.empty(d["sum_cig"], np.uint32), np.empty(n + 1, np.uint32), np.empty(d["sum_seq"], np.uint8),
                      np.empty(n + 1, np.uint32), np.empty(d["sum_qual"], np.uint8))
        rec_off = np.empty(n, np.uint64)
        bo = AmpBatchOut(_ptr(b.pos), _ptr(b.flag), _ptr(b.tlen), _ptr(b.cig_off), _ptr(b.cigar), _ptr(b.seq_off), _ptr(b.seq),
                         _ptr(b.qual_off), _ptr(b.qual))
        _check(self.lib.amp_decoded_copy_host(self._ctx, ctypes.byref(bo), _ptr(rec_off)), "amp_decoded_copy_host")
        return b, rec_off

    def decoded_write_bam(self, header_bytes):
        """The trimmed BAM file (uint8 array) of the batch decode_bam + process_decoded(trim=True) left in HBM, and the number of
        records in it (amp_decoded_write_bam); ``header_bytes``: the BAM header the file starts with."""
        hb = np.frombuffer(header_bytes, np.uint8) if not isinstance(header_bytes, np.ndarray) else header_bytes
        raw = int(self._decoded["raw_bytes"])
        out = np.empty(hb.size + raw + raw // 1000 + 4 * int(self._decoded["sum_cig"]) + 12 * int(self._decoded["n"]) + 4096, np.uint8)
        nrec = ctypes.c_int64(0)
        self.lib.amp_decoded_write_bam.restype = ctypes.c_int64
        r = int(self.lib.amp_decoded_write_bam(self._ctx, _ptr(hb), ctypes.c_int64(hb.size), _ptr(out), ctypes.c_int64(out.size), ctypes.byref(nrec)))
        if r < 0:
            _check(r, "amp_decoded_write_bam")
        self.launches += 5
        return out[:r], int(nrec.value)

    def bgzf_deflate(self, data, bstart):
        """BGZF blocks (+ EOF block) of ``data`` cut at ``bstart`` (n_blocks + 1 offsets, each block <= 0xff00 bytes), compressed
        on the device (amp_bgzf_deflate_host).  Returns a uint8 array."""
        src = np.ascontiguousarray(data, np.uint8)
        bs = np.ascontiguousarray(bstart, np.int64)
        nb = bs.size - 1
        out = np.empty(src.size + 31 * max(nb, 0) + 28, np.uint8)
        self.lib.amp_bgzf_deflate_host.restype = ctypes.c_int64
        r = int(self.lib.amp_bgzf_deflate_host(self._ctx, _ptr(src), ctypes.c_int64(src.size), _ptr(bs), ctypes.c_int64(nb), _ptr(out),
                                               ctypes.c_int64(out.size)))
        if r < 0:
            _check(r, "amp_bgzf_deflate_host")
        self.launches += 2
        return out[:r]

    # ---------------------------------------------------------------- deep-sample exchange (dist.py)
    def reserve(self, max_reads, max_cigar_ops):
        """Pre-size the buffers process_device would otherwise grow on demand (no allocation on the hot path afterwards)."""
        _check(self.lib.amp_reserve(self._ctx, ctypes.c_int64(int(max_reads)), ctypes.c_int64(int(max_cigar_ops))), "amp_reserve")

    def allreduce_counts(self, comm, stream=None):
        """One ncclAllReduce(sum, int32) of the count matrices, in place (``comm``: NcclComm or a raw ncclComm_t value)."""
        h = comm.handle if hasattr(comm, "handle") else comm
        _check(self.lib.amp_allreduce_counts(self._ctx, ctypes.c_void_p(h), ctypes.c_void_p(stream) if stream else None),
               "amp_allreduce_counts")

    def ins_slot_bytes(self, cap_entries, cap_arena_bytes):
        return int(self.lib.amp_ins_slot_bytes(ctypes.c_int64(cap_entries), ctypes.c_int64(cap_arena_bytes)))

    def ins_pack_device(self, dev_ptr, cap_entries, cap_arena_bytes, stream=None):
        _check(self.lib.amp_ins_pack_device(self._ctx, ctypes.c_void_p(dev_ptr), ctypes.c_int64(cap_entries),
                                            ctypes.c_int64(cap_arena_bytes), ctypes.c_void_p(stream) if stream else None),
               "amp_ins_pack_device")
        self.launches += 1

    def ins_merge_packed(self, dev_ptr, n_ranks, my_rank, cap_entries, cap_arena_bytes, stream=None):
        _check(self.lib.amp_ins_merge_packed(self._ctx, ctypes.c_void_p(dev_ptr), int(n_ranks), int(my_rank),
                                             ctypes.c_int64(cap_entries), ctypes.c_int64(cap_arena_bytes),
                                             ctypes.c_void_p(stream) if stream else None), "amp_ins_merge_packed")
        self.launches += 1

    # the same exchange for a context with the strand / quality sums (enable_qstats): the methods above refuse such a context
    def allreduce_qstats(self, comm, stream=None):
        """ncclAllReduce(sum) of the counts, rev and qsum matrices, in place (``comm``: NcclComm or a raw ncclComm_t value)."""
        h = comm.handle if hasattr(comm, "handle") else comm
        _check(self.lib.amp_allreduce_qstats(self._ctx, ctypes.c_void_p(h), ctypes.c_void_p(stream) if stream else None),
               "amp_allreduce_qstats")

    def ins_slot_bytes_qstats(self, cap_entries, cap_arena_bytes):
        return int(self.lib.amp_ins_slot_bytes_qstats(ctypes.c_int64(cap_entries), ctypes.c_int64(cap_arena_bytes)))

    def ins_pack_qstats_device(self, dev_ptr, cap_entries, cap_arena_bytes, stream=None):
        _check(self.lib.amp_ins_pack_qstats_device(self._ctx, ctypes.c_void_p(dev_ptr), ctypes.c_int64(cap_entries),
                                                   ctypes.c_int64(cap_arena_bytes), ctypes.c_void_p(stream) if stream else None),
               "amp_ins_pack_qstats_device")
        self.launches += 1

    def ins_merge_packed_qstats(self, dev_ptr, n_ranks, my_rank, cap_entries, cap_arena_bytes, stream=None):
        _check(self.lib.amp_ins_merge_packed_qstats(self._ctx, ctypes.c_void_p(dev_ptr), int(n_ranks), int(my_rank),
                                                    ctypes.c_int64(cap_entries), ctypes.c_int64(cap_arena_bytes),
                                                    ctypes.c_void_p(stream) if stream else None), "amp_ins_merge_packed_qstats")
        self.launches += 1

    # ---------------------------------------------------------------- iVar-format outputs (DESIGN.md 3.7)
    def enable_qstats(self):
        """Allocate the strand / quality sums (amp_qstats_enable); process(..., qstats=True) fills them."""
        _check(self.lib.amp_qstats_enable(self._ctx), "amp_qstats_enable")
        self._qstats = True

    @property
    def qstats_enabled(self):
        """True once enable_qstats has succeeded: the context holds the strand / quality sums."""
        return self._qstats

    def qstats(self, sample=0):
        """The strand / quality sums of one sample: rev / qsum [6, L] and, in insertions() order (all samples), ins_rev /
        ins_qsum / ins_head."""
        n = ctypes.c_int64(0)
        nch = ctypes.c_int64(0)
        _check(self.lib.amp_ins_count(self._ctx, ctypes.byref(n), ctypes.byref(nch)), "amp_ins_count")
        k = int(n.value)
        q = QStats(np.empty((6, self.L), np.int32), np.empty((6, self.L), np.int64), np.zeros(max(k, 1), np.int32),
                   np.zeros(max(k, 1), np.int64), np.zeros(max(k, 1), np.uint8))
        _check(self.lib.amp_qstats_host(self._ctx, int(sample), _ptr(q.rev), _ptr(q.qsum), _ptr(q.ins_rev), _ptr(q.ins_qsum),
                                        _ptr(q.ins_head)), "amp_qstats_host")
        q.ins_rev, q.ins_qsum, q.ins_head = q.ins_rev[:k], q.ins_qsum[:k], q.ins_head[:k]
        return q

    def call_ivar(self, min_depth=1, min_freq=0.03, iupac_threshold=0.0):
        """Mean qualities, Fisher p-values and IUPAC codes (amp_call_ivar) on the outputs of the last ``call``."""
        n = ctypes.c_int64(0)
        nch = ctypes.c_int64(0)
        _check(self.lib.amp_ins_count(self._ctx, ctypes.byref(n), ctypes.byref(nch)), "amp_ins_count")
        k = max(int(n.value), 1)
        SL = self.n_samples * self.L
        r = IvarResult(np.empty(SL, np.uint8), np.empty((SL, 6), np.int32), np.empty((SL, 6), np.float64), np.zeros(k, np.int32),
                       np.full(k, np.nan))
        p = AmpIvarParams(int(min_depth), float(min_freq), float(iupac_threshold))
        _check(self.lib.amp_call_ivar(self._ctx, ctypes.byref(p), _ptr(r.iupac), _ptr(r.fixed_mq), _ptr(r.fixed_pval),
                                      _ptr(r.ins_mq), _ptr(r.ins_pval)), "amp_call_ivar")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return r

    def call_ivar_device(self, min_depth=1, min_freq=0.03, iupac_threshold=0.0, stream=None):
        p = AmpIvarParams(int(min_depth), float(min_freq), float(iupac_threshold))
        _check(self.lib.amp_call_ivar_device(self._ctx, ctypes.byref(p), ctypes.c_void_p(stream) if stream else None),
               "amp_call_ivar_device")
        self.launches += int(self.lib.amp_last_launches(self._ctx))

    # ---------------------------------------------------------------- anchored deletion alleles of the iVar TSV (DESIGN.md 3.7)
    def enable_dels(self, slots=0):
        """Allocate the anchored deletion table (amp_dels_enable; ``slots`` a power of two, 0 = 2^20) after enable_qstats;
        process(..., qstats=True) fills it."""
        _check(self.lib.amp_dels_enable(self._ctx, ctypes.c_int64(int(slots))), "amp_dels_enable")
        self._dels = True

    @property
    def dels_enabled(self):
        """True once enable_dels has succeeded."""
        return self._dels

    def dels(self, sample=None):
        """The anchored deletion alleles sorted by (sample, anchor, len) (amp_dels_export); ``sample``: only that sample's."""
        n = ctypes.c_int64(0)
        _check(self.lib.amp_dels_count(self._ctx, ctypes.byref(n)), "amp_dels_count")
        k = int(n.value)
        d = Deletions(*[np.zeros(max(k, 1), t) for t in (np.int32,) * 5 + (np.int64,)])
        _check(self.lib.amp_dels_export(self._ctx, _ptr(d.sample), _ptr(d.anchor), _ptr(d.len), _ptr(d.count), _ptr(d.rev), _ptr(d.qsum)),
               "amp_dels_export")
        d = d.take(np.arange(k))
        return d if sample is None else d.take(np.flatnonzero(d.sample == sample))

    def merge_dels(self, d):
        """Add the alleles of a Deletions (e.g. another rank's) to the table: the host form of the exchange."""
        a = [np.ascontiguousarray(x, t) for x, t in ((d.sample, np.int32), (d.anchor, np.int32), (d.len, np.int32), (d.count, np.int32),
                                                     (d.rev, np.int32), (d.qsum, np.int64))]
        _check(self.lib.amp_dels_merge(self._ctx, ctypes.c_int64(len(a[0])), *[_ptr(x) for x in a]), "amp_dels_merge")
        self.launches += 1

    def call_ivar_dels(self, min_depth=1, min_freq=0.03):
        """The alleles of ``dels()`` with mq and PVAL (amp_call_ivar_dels; NaN = no TSV row), on the depths of the last ``call``."""
        d = self.dels()
        k = len(d.count)
        mq, pval = np.zeros(max(k, 1), np.int32), np.full(max(k, 1), np.nan)
        p = AmpIvarParams(int(min_depth), float(min_freq), 0.0)
        _check(self.lib.amp_call_ivar_dels(self._ctx, ctypes.byref(p), _ptr(mq), _ptr(pval)), "amp_call_ivar_dels")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        d.mq, d.pval = mq[:k], pval[:k]
        return d

    def dels_slot_bytes(self, cap_entries):
        return int(self.lib.amp_dels_slot_bytes(ctypes.c_int64(cap_entries)))

    def dels_pack_device(self, dev_ptr, cap_entries, stream=None):
        _check(self.lib.amp_dels_pack_device(self._ctx, ctypes.c_void_p(dev_ptr), ctypes.c_int64(cap_entries),
                                             ctypes.c_void_p(stream) if stream else None), "amp_dels_pack_device")
        self.launches += 1

    def dels_merge_packed(self, dev_ptr, n_ranks, my_rank, cap_entries, stream=None):
        _check(self.lib.amp_dels_merge_packed(self._ctx, ctypes.c_void_p(dev_ptr), int(n_ranks), int(my_rank), ctypes.c_int64(cap_entries),
                                              ctypes.c_void_p(stream) if stream else None), "amp_dels_merge_packed")
        self.launches += 1

    # ---------------------------------------------------------------- codon annotation of the iVar TSV (DESIGN.md 3.9)
    def set_features(self, sample, features):
        """The CDS features of one sample (gff.Feature: strand, phase, segments); checked against the sample's reference, which
        has to be set first (set_reference / set_sample_reference / call).  An empty list clears the sample."""
        strand = np.ascontiguousarray([f.strand for f in features], np.int32)
        phase = np.ascontiguousarray([f.phase for f in features], np.int32)
        seg_off = np.zeros(len(features) + 1, np.int32)
        np.cumsum([len(f.segments) for f in features], out=seg_off[1:])
        start = np.ascontiguousarray([s for f in features for s, _ in f.segments], np.int32)
        end = np.ascontiguousarray([e for f in features for _, e in f.segments], np.int32)
        _check(self.lib.amp_set_features(self._ctx, int(sample), len(features), _ptr(strand), _ptr(phase), _ptr(seg_off), _ptr(start),
                                         _ptr(end)), "amp_set_features")

    def annotate(self):
        """The occurrences of every (sample, position) in the features of set_features, built and translated on the device
        (amp_annotate + amp_annot_host).  Returns an ivar.Annotation."""
        n = ctypes.c_int64(0)
        _check(self.lib.amp_annotate(self._ctx, ctypes.byref(n)), "amp_annotate")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        E = int(n.value)
        a = Annotation(self.L, np.empty(self.n_samples * self.L + 1, np.uint32), np.empty(max(E, 1), np.int32), np.empty(max(E, 1), np.int32),
                       np.empty(max(E, 1), np.uint8), np.empty((max(E, 1), 18), np.uint8), np.empty((max(E, 1), 6), np.uint8))
        _check(self.lib.amp_annot_host(self._ctx, _ptr(a.off), _ptr(a.feat), _ptr(a.pos_aa), _ptr(a.codon_off), _ptr(a.codons), _ptr(a.aas)),
               "amp_annot_host")
        a.feat, a.pos_aa, a.codon_off, a.codons, a.aas = a.feat[:E], a.pos_aa[:E], a.codon_off[:E], a.codons[:E], a.aas[:E]
        return a

    def _call_buffers(self, n_ins, pinned):
        """Result arrays of ``call``: fresh numpy arrays, or (``pinned``) page-locked arrays owned by the engine and reused."""
        SL = self.n_samples * self.L
        K = max(n_ins, 1)
        spec = [((SL,), np.int32), ((SL,), np.int32), ((SL,), np.int32), ((SL,), np.uint8), ((SL,), np.int32),
                ((SL, 6), np.float64), ((SL, 6), np.int32), ((SL,), np.uint8), ((K,), np.float64), ((K,), np.int32),
                ((K,), np.uint8)]
        if not pinned:
            return [np.empty(sh, dt) if i < 8 else np.zeros(sh, dt) for i, (sh, dt) in enumerate(spec)]
        import torch
        cache = getattr(self, "_pinned_call", None)
        if cache is None or cache[0] < K:
            cap = max(K, 1024) * 2 if cache is not None else max(K, 1024)
            tens = [torch.zeros(sh if i < 8 else (cap,), dtype=getattr(torch, np.dtype(dt).name), pin_memory=True)
                    for i, (sh, dt) in enumerate(spec)]
            cache = self._pinned_call = (cap, tens)
        arrs = [t.numpy() for t in cache[1]]
        for a in arrs[8:]:
            a[:K] = 0
        return arrs[:8] + [a[:K] for a in arrs[8:]]

    def call(self, ref_seq, min_depth_consensus=10, min_freq_consensus=0.0, min_depth_variants=1,
             min_freq_variants=0.03, n_ins=None, pinned=False):
        """``pinned=True``: the result arrays are page-locked buffers owned by the engine (the device-to-host copies run
        at full PCIe speed) and stay valid until the next ``call`` on this engine."""
        if n_ins is None:
            n = ctypes.c_int64(0)
            nch = ctypes.c_int64(0)
            _check(self.lib.amp_ins_count(self._ctx, ctypes.byref(n), ctypes.byref(nch)), "amp_ins_count")
            n_ins = int(n.value)
        r = CallResult(self.L, self.n_samples, *self._call_buffers(n_ins, pinned))
        co = AmpCallOut(_ptr(r.depth), _ptr(r.top_id), _ptr(r.top_count), _ptr(r.pos_flags), _ptr(r.ref_count),
                        _ptr(r.fixed_freq), _ptr(r.fixed_rank), _ptr(r.alt_mask))
        cp = AmpCallParams(int(min_depth_consensus), float(min_freq_consensus), int(min_depth_variants),
                           float(min_freq_variants))
        if ref_seq is None:      # keep the reference uploaded by set_reference()
            ref_arg = None
        else:
            ref = ref_seq.encode("latin-1") if isinstance(ref_seq, str) else bytes(ref_seq)
            assert len(ref) == self.L
            ref_arg = ctypes.c_char_p(ref)
        _check(self.lib.amp_call(self._ctx, ref_arg, ctypes.byref(cp), ctypes.byref(co), _ptr(r.ins_freq),
                                 _ptr(r.ins_rank), _ptr(r.ins_alt)), "amp_call")
        self.launches += int(self.lib.amp_last_launches(self._ctx))
        return r


class NcclComm:
    """An ncclComm_t created through the C ABI (amp_nccl_unique_id / amp_nccl_comm_init).  The 128-byte id of rank 0 has
    to reach the other ranks somehow; ``from_torch_group`` broadcasts it over an initialised torch.distributed group."""

    def __init__(self, handle, rank, world):
        self.handle, self.rank, self.world = handle, rank, world

    @staticmethod
    def unique_id():
        buf = (ctypes.c_uint8 * 128)()
        _check(load_library().amp_nccl_unique_id(buf), "amp_nccl_unique_id")
        return bytes(buf)

    @classmethod
    def create(cls, device, world, rank, unique_id):
        assert len(unique_id) == 128
        h = ctypes.c_void_p()
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(load_library().amp_nccl_comm_init(int(device), int(world), int(rank), buf, ctypes.byref(h)), "amp_nccl_comm_init")
        return cls(h.value, rank, world)

    @classmethod
    def from_torch_group(cls, device, group=None):
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        uid = cls.unique_id() if rank == 0 else bytes(128)
        t = torch.tensor(list(uid), dtype=torch.uint8, device=torch.device("cuda", device) if dist.get_backend(group) == "nccl" else "cpu")
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        return cls.create(device, world, rank, bytes(t.cpu().tolist()))

    def allgather(self, send_ptr, recv_ptr, bytes_per_rank, stream=None):
        _check(load_library().amp_nccl_allgather(ctypes.c_void_p(self.handle), ctypes.c_void_p(send_ptr), ctypes.c_void_p(recv_ptr),
                                                 ctypes.c_int64(bytes_per_rank), ctypes.c_void_p(stream) if stream else None),
               "amp_nccl_allgather")

    def close(self):
        if self.handle:
            load_library().amp_nccl_comm_destroy(ctypes.c_void_p(self.handle))
            self.handle = None
