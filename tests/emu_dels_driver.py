"""TEST INFRASTRUCTURE: emu_dist_driver.EmuQstatsEngine with the Engine surface of the anchored deletion alleles, backed by
tests/emu/amp_emu_dels.cpp (the kernels' own source, amp_dels.cuh included, compiled for the CPU).

The library is a superset of emu_dist_driver's: ``install`` routes emu_driver's and emu_dist_driver's calls to it, so one context
sees one emulator."""
import ctypes
import glob
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import emu_dist_driver
import emu_driver
from amplipy_b200.ivar import Deletions

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
_p = emu_driver._p


def build():
    """g++ amp_emu_dels.cpp -> a shared library in the temporary directory, keyed by the sources (the tree may be read-only)."""
    srcs = sorted(glob.glob(os.path.join(_HERE, "emu", "amp_emu*.cpp")) + glob.glob(os.path.join(_HERE, "..", "amplipy_b200", "csrc", "*.cuh")))
    key = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
    so = os.path.join(tempfile.gettempdir(), "amplipy_b200_emu_dels_%d_%s.so" % (os.getuid(), key))
    if not os.path.isfile(so):
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2", "-o", tmp,
                               os.path.join(_HERE, "emu", "amp_emu_dels.cpp")])
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
        lb.emu_dels_count.restype = ctypes.c_longlong
        lb.emu_dels_home.restype = ctypes.c_ulonglong
        lb.emu_dels_home.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_longlong]
        lb.emu_fisher_less.restype = ctypes.c_double
        lb.emu_fisher_less.argtypes = [ctypes.c_longlong, ctypes.c_longlong, ctypes.c_int]
        _lib = lb
    return _lib


def install(monkeypatch=None):
    """Route emu_driver's and emu_dist_driver's library calls to this library (``monkeypatch``: for the duration of a test)."""
    get = lambda: lib()
    for m in (emu_driver, emu_dist_driver):
        if monkeypatch is not None:
            monkeypatch.setattr(m, "lib", get)
        else:
            m.lib = get


def home_slot(gpos, length, slots):
    """The slot at which the probe of allele (gpos = sample * lpad + anchor, length) starts in a table of ``slots`` slots."""
    return int(lib().emu_dels_home(int(gpos), int(length), int(slots)))


class EmuDelsEngine(emu_dist_driver.EmuQstatsEngine):
    """EmuQstatsEngine plus enable_dels / dels / merge_dels / call_ivar_dels, reset of the table, and the emulated pack / merge.
    Needs ``install`` first."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self._dels = False

    @property
    def dels_enabled(self):
        return self._dels

    def enable_dels(self, slots=0):
        assert self._qstats, "enable_dels needs enable_qstats"
        n = int(slots) or (1 << 20)
        lib().emu_dels_enable(self._h, ctypes.c_longlong(1 << (n - 1).bit_length()))
        self._dels = True

    def process(self, batch, trim=True, pileup=True, sample=0, first=0, n=None, qstats=False):
        if not (qstats and self._dels):
            return super().process(batch, trim=trim, pileup=pileup, sample=sample, first=first, n=n, qstats=qstats)
        t = emu_driver.EmuEngine.process(self, batch, trim=trim, pileup=pileup, sample=sample, first=first, n=n)
        assert self._qstats and pileup
        n = batch.n - first if n is None else n
        o = (None,) * 4 if t is None else (t.pos, t.ncig, t.flags, t.cigar)
        lib().emu_qstats_dels_pass(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag), _p(batch.tlen),
                                   _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(batch.seq), _p(batch.qual_off), _p(batch.qual),
                                   1 if trim else 0, sample, *[_p(a) for a in o])
        return t

    def reset(self):
        super().reset()
        if self._dels:
            lib().emu_dels_reset(self._h)

    def dels(self, sample=None):
        k = int(lib().emu_dels_count(self._h))
        d = Deletions(*[np.zeros(max(k, 1), t) for t in (np.int32,) * 5 + (np.int64,)])
        lib().emu_dels_export(self._h, _p(d.sample), _p(d.anchor), _p(d.len), _p(d.count), _p(d.rev), _p(d.qsum))
        d = d.take(np.arange(k))
        return d if sample is None else d.take(np.flatnonzero(d.sample == sample))

    def merge_dels(self, d):
        a = [np.ascontiguousarray(x, t) for x, t in ((d.sample, np.int32), (d.anchor, np.int32), (d.len, np.int32), (d.count, np.int32),
                                                     (d.rev, np.int32), (d.qsum, np.int64))]
        lib().emu_dels_merge(self._h, ctypes.c_longlong(len(a[0])), *[_p(x) for x in a])

    def call_ivar_dels(self, min_depth=1, min_freq=0.03):
        d = self.dels()
        k = len(d.count)
        mq, pval = np.zeros(max(k, 1), np.int32), np.full(max(k, 1), np.nan)
        lib().emu_call_ivar_dels(self._h, _p(self._res.depth), int(min_depth), ctypes.c_double(min_freq), _p(mq), _p(pval))
        d.mq, d.pval = mq[:k], pval[:k]
        return d

    @staticmethod
    def dels_slot_bytes(cap_entries):
        return 8 + 32 * int(cap_entries)

    def dels_pack(self, slot, cap_entries):
        assert slot.dtype == np.uint64 and slot.flags.c_contiguous and slot.nbytes >= self.dels_slot_bytes(cap_entries)
        lib().emu_dels_pack(self._h, _p(slot), ctypes.c_longlong(cap_entries))

    def dels_merge_packed(self, slots, n_ranks, my_rank, cap_entries):
        assert slots.dtype == np.uint64 and slots.flags.c_contiguous and slots.nbytes >= n_ranks * self.dels_slot_bytes(cap_entries)
        lib().emu_dels_merge_packed(self._h, _p(slots), int(n_ranks), int(my_rank), ctypes.c_longlong(cap_entries))
