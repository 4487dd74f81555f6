"""TEST INFRASTRUCTURE: emu_driver.EmuEngine with the Engine surface of the strand / quality sums and their deep-sample exchange,
backed by tests/emu/amp_emu_dist.cpp (the kernels' own source, amp_ivar.cuh and amp_exchange.cuh included, compiled for the CPU).

The library is a superset of emu_driver's: ``install`` routes emu_driver's calls to it, so one context sees one emulator."""
import ctypes
import glob
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import emu_driver
from amplipy_b200.ivar import IvarResult, QStats

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_p = emu_driver._p


def build():
    """g++ amp_emu_dist.cpp -> a shared library in the temporary directory, keyed by the sources (the tree may be read-only)."""
    srcs = sorted(glob.glob(os.path.join(_HERE, "emu", "amp_emu*.cpp")) + glob.glob(os.path.join(_HERE, "..", "amplipy_b200", "csrc", "*.cuh")))
    key = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "amplipy_b200_emu_dist_%d_%s.so" % (os.getuid(), key))
    if not os.path.isfile(so):
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2", "-o", tmp,
                               os.path.join(_HERE, "emu", "amp_emu_dist.cpp")])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        lb = ctypes.CDLL(build())
        lb.emu_create.restype = ctypes.c_void_p
        lb.emu_ins_count.restype = ctypes.c_longlong
        lb.emu_ins_chars.restype = ctypes.c_longlong
        lb.emu_error_flags.restype = ctypes.c_uint
        lb.emu_ins_hash.restype = ctypes.c_ulonglong
        lb.emu_ins_hash.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
        lb.emu_rev_ptr.restype = ctypes.POINTER(ctypes.c_int32)
        lb.emu_qsum_ptr.restype = ctypes.POINTER(ctypes.c_int64)
        _lib = lb
    return _lib


def install(monkeypatch=None):
    """Route emu_driver's library calls to this library (``monkeypatch``: for the duration of a test)."""
    get = lambda: lib()
    if monkeypatch is not None:
        monkeypatch.setattr(emu_driver, "lib", get)
    else:
        emu_driver.lib = get


class EmuQstatsEngine(emu_driver.EmuEngine):
    """EmuEngine plus enable_qstats / process(..., qstats=True) / qstats / call_ivar, tensors over the emulated rev / qsum, merges that
    carry the sums, and the emulated stats pack / merge.  Needs ``install`` first."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._qstats = False

    @property
    def qstats_enabled(self):
        return self._qstats

    def enable_qstats(self):
        lib().emu_qstats_enable(self._h)
        self._qstats = True

    def process(self, batch, trim=True, pileup=True, sample=0, first=0, n=None, qstats=False):
        """``qstats=True``: the strand / quality pass (emu_qstats_pass) on the same reads after the fused kernel."""
        t = super().process(batch, trim=trim, pileup=pileup, sample=sample, first=first, n=n)
        if qstats:
            assert self._qstats and pileup, "qstats needs enable_qstats and pileup"
            n = batch.n - first if n is None else n
            o = (None,) * 4 if t is None else (t.pos, t.ncig, t.flags, t.cigar)
            lib().emu_qstats_pass(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag), _p(batch.tlen),
                                  _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(batch.seq), _p(batch.qual_off), _p(batch.qual),
                                  1 if trim else 0, sample, *[_p(a) for a in o])
        return t

    def qstats(self, sample=0):
        k = int(lib().emu_ins_count(self._h))
        q = QStats(np.empty((6, self.L), np.int32), np.empty((6, self.L), np.int64), np.zeros(max(k, 1), np.int32),
                   np.zeros(max(k, 1), np.int64), np.zeros(max(k, 1), np.uint8))
        lib().emu_qstats_host(self._h, sample, _p(q.rev), _p(q.qsum), _p(q.ins_rev), _p(q.ins_qsum), _p(q.ins_head))
        q.ins_rev, q.ins_qsum, q.ins_head = q.ins_rev[:k], q.ins_qsum[:k], q.ins_head[:k]
        return q

    def qstats_tensors(self):
        """(rev int32, qsum int64) tensors [n_samples, 6, lpad] over the emulated sums, as counts_tensor is over the counts (qsum holds
        uint64 sums; int64 adds them to the same bits)."""
        import torch
        shape = (self.n_samples, 6, int(lib().emu_lpad(self._h)))
        return (torch.from_numpy(np.ctypeslib.as_array(lib().emu_rev_ptr(self._h), shape=shape)),
                torch.from_numpy(np.ctypeslib.as_array(lib().emu_qsum_ptr(self._h), shape=shape)))

    def call(self, ref_seq, *a, **kw):
        self._ref = ref_seq
        self._res = super().call(ref_seq, *a, **kw)
        return self._res

    def call_ivar(self, min_depth=1, min_freq=0.03, iupac_threshold=0.0):
        """emu_call_ivar on the outputs of the last ``call``."""
        r = self._res
        k = max(int(lib().emu_ins_count(self._h)), 1)
        SL = self.n_samples * self.L
        out = IvarResult(np.empty(SL, np.uint8), np.empty((SL, 6), np.int32), np.empty((SL, 6), np.float64), np.zeros(k, np.int32),
                         np.full(k, np.nan))
        lib().emu_call_ivar(self._h, ctypes.c_char_p(self._ref.encode("latin-1")), _p(r.depth), _p(r.top_id), _p(r.top_count),
                            _p(r.fixed_freq), _p(r.fixed_rank), _p(r.ins_freq), _p(r.ins_rank), int(min_depth), ctypes.c_double(min_freq),
                            ctypes.c_double(iupac_threshold), _p(out.iupac), _p(out.fixed_mq), _p(out.fixed_pval), _p(out.ins_mq),
                            _p(out.ins_pval))
        return out

    def merge_insertions(self, sample, pos, count, str_off, chars, ins_rev=None, ins_qsum=None, ins_head=None):
        """Add alleles to the table; with ``ins_rev`` / ``ins_qsum`` / ``ins_head`` their strand / quality sums too."""
        if ins_rev is None:
            return super().merge_insertions(sample, pos, count, str_off, chars)
        assert self._qstats
        chars = np.ascontiguousarray(chars, np.uint8) if len(chars) else np.zeros(1, np.uint8)
        lib().emu_ins_merge_qstats(self._h, ctypes.c_longlong(len(pos)), _p(np.ascontiguousarray(sample, np.int32)),
                                   _p(np.ascontiguousarray(pos, np.int32)), _p(np.ascontiguousarray(count, np.int32)),
                                   _p(np.ascontiguousarray(str_off, np.int64)), _p(chars), _p(np.ascontiguousarray(ins_rev, np.int32)),
                                   _p(np.ascontiguousarray(ins_qsum, np.int64)), _p(np.ascontiguousarray(ins_head, np.uint8)))

    @staticmethod
    def ins_slot_bytes_qstats(cap_entries, cap_arena_bytes):
        return 16 + 32 * int(cap_entries) + ((int(cap_arena_bytes) + 7) & ~7)

    def ins_pack_qstats(self, slot, cap_entries, cap_arena_bytes):
        """The table with its sums packed into ``slot`` (a uint64 array of ins_slot_bytes_qstats / 8 words)."""
        assert slot.dtype == np.uint64 and slot.flags.c_contiguous and slot.nbytes >= self.ins_slot_bytes_qstats(cap_entries, cap_arena_bytes)
        lib().emu_ins_pack_qstats(self._h, _p(slot), ctypes.c_longlong(cap_entries), ctypes.c_longlong(cap_arena_bytes))

    def ins_merge_packed_qstats(self, slots, n_ranks, my_rank, cap_entries, cap_arena_bytes):
        """Every slot of ``slots`` (n_ranks of them, back to back) except my_rank's merged into the table with its sums."""
        assert slots.dtype == np.uint64 and slots.flags.c_contiguous
        assert slots.nbytes >= n_ranks * self.ins_slot_bytes_qstats(cap_entries, cap_arena_bytes)
        lib().emu_ins_merge_packed_qstats(self._h, _p(slots), int(n_ranks), int(my_rank), ctypes.c_longlong(cap_entries),
                                          ctypes.c_longlong(cap_arena_bytes))
