"""TEST INFRASTRUCTURE: same surface as amplipy_b200.engine.Engine, backed by tests/emu (the kernels'
own source compiled for the CPU).  Lets the build container exercise the device logic without a GPU."""
import ctypes
import os
import subprocess

import numpy as np

from amplipy_b200.calling import CallResult, Insertions
from amplipy_b200.engine import TrimResult

_HERE = os.path.dirname(os.path.abspath(__file__))
_DIR = os.path.join(_HERE, "emu")
_lib = None


def build(asan=False):
    name = "libamp_emu_asan.so" if asan else "libamp_emu.so"
    so = os.path.join(_DIR, name)
    srcs = [os.path.join(_DIR, "amp_emu.cpp"), os.path.join(_HERE, "..", "amplipy_b200", "csrc", "amp_core.cuh"),
            os.path.join(_HERE, "..", "amplipy_b200", "csrc", "amp_kernels.cuh"),
            os.path.join(_HERE, "..", "amplipy_b200", "csrc", "amp_warp.cuh"),
            os.path.join(_HERE, "..", "amplipy_b200", "csrc", "amp_bgzf.cuh"),
            os.path.join(_HERE, "..", "amplipy_b200", "csrc", "amp_ont.cuh")]
    if not os.path.isfile(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        flags = ["-O1", "-g", "-fsanitize=address,undefined"] if asan else ["-O2"]
        subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable"] + flags +
                              ["-o", so, srcs[0]])
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build(asan=bool(os.environ.get("AMP_EMU_ASAN"))))
        _lib.emu_create.restype = ctypes.c_void_p
        _lib.emu_ins_count.restype = ctypes.c_longlong
        _lib.emu_ins_chars.restype = ctypes.c_longlong
        _lib.emu_error_flags.restype = ctypes.c_uint
        _lib.emu_ins_hash.restype = ctypes.c_ulonglong
        _lib.emu_ins_hash.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    return _lib


def ins_hash(gpos, text):
    """The 64-bit hash ins_table_add computes for the insertion key ``text`` at ``gpos`` (sample * lpad + pos)."""
    raw = text.encode("latin-1")
    return int(lib().emu_ins_hash(int(gpos), raw, len(raw)))


def v7_stats(reset=True):
    """(reads finished on the cooperative path, reads sent to the generic path) since the last reset."""
    out = (ctypes.c_longlong * 2)()
    lib().emu_v7_stats(out, 1 if reset else 0)
    return int(out[0]), int(out[1])


def _p(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


class EmuEngine:
    def __init__(self, ref_len, primer_tables=None, max_primer_len=0, min_quality=20, sliding_window_width=4,
                 min_length=30, include_no_primer=False, n_samples=1, ins_slots=1 << 16, ins_arena_bytes=1 << 22, device=0,
                 grid=0, threads=256, reads_per_tile=0, maxseg=0, wt=0, qbytes=0, kernel="tile", warps=0, batch_reads=0):
        self.L, self.n_samples = int(ref_len), int(n_samples)
        ins_slots = min(ins_slots or (1 << 16), 1 << 18)
        ins_arena_bytes = min(ins_arena_bytes or (1 << 22), 1 << 24)
        mn = mx = None
        if primer_tables is not None:
            mn = np.ascontiguousarray(primer_tables[0], np.int32)
            mx = np.ascontiguousarray(primer_tables[1], np.int32)
        self._h = ctypes.c_void_p(lib().emu_create(self.L, n_samples, _p(mn), _p(mx), int(max_primer_len), min_quality,
                                                   sliding_window_width, min_length, 1 if include_no_primer else 0,
                                                   ctypes.c_longlong(ins_slots), ctypes.c_longlong(ins_arena_bytes)))
        self.knobs = (grid, threads, reads_per_tile, maxseg, wt, qbytes)
        # kernel="v7": the warp-autonomous kernel of amp_warp.cuh (every CUDA thread a fiber); "tile": amp_kernels.cuh
        self.kernel, self.v7_knobs = kernel, (grid, warps, batch_reads, wt)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().emu_destroy(self._h)
            self._h = None

    def error_flags(self):
        return int(lib().emu_error_flags(self._h))

    def reset(self):
        lib().emu_reset(self._h)

    def raise_on_device_errors(self):
        assert self.error_flags() == 0, self.error_flags()

    def process(self, batch, trim=True, pileup=True, sample=0, first=0, n=None):
        n = batch.n - first if n is None else n
        out = (np.zeros(batch.n, np.int32), np.zeros(batch.n, np.uint16), np.zeros(batch.n, np.uint8),
               np.zeros(int(batch.cig_off[-1]) + 3 * batch.n, np.uint32))
        mode = (1 if trim else 0) | (2 if pileup else 0)
        # the staging loops read 16-byte vectors from 16-byte aligned addresses: keep numpy buffers aligned
        qual = _aligned(batch.qual)
        seq = _aligned(batch.seq)
        if self.kernel == "ont":
            g, w, br, wt = self.v7_knobs
            lib().emu_process_ont(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag),
                                  _p(batch.tlen), _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(seq),
                                  _p(batch.qual_off), _p(qual), mode, sample, _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]),
                                  g, w, wt)
            return TrimResult(batch, *out) if trim else None
        if self.kernel == "v7":
            g, w, br, wt = self.v7_knobs
            lib().emu_process_v7(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag),
                                 _p(batch.tlen), _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(seq),
                                 _p(batch.qual_off), _p(qual), mode, sample, _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]),
                                 g, w, br, wt)
            return TrimResult(batch, *out) if trim else None
        g, t, r, ms, wt, qb = self.knobs
        lib().emu_process(self._h, ctypes.c_longlong(first), ctypes.c_longlong(n), _p(batch.pos), _p(batch.flag),
                          _p(batch.tlen), _p(batch.cig_off), _p(batch.cigar), _p(batch.seq_off), _p(seq),
                          _p(batch.qual_off), _p(qual), mode, sample, _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]),
                          g, t, r, ms, wt, qb)
        return TrimResult(batch, *out) if trim else None

    def counts(self, sample=0):
        out = np.empty((6, self.L), np.int32)
        lib().emu_counts(self._h, sample, _p(out))
        return out

    def counts_tensor(self):
        import torch
        lib().emu_counts_ptr.restype = ctypes.POINTER(ctypes.c_int)
        lpad = int(lib().emu_lpad(self._h))
        arr = np.ctypeslib.as_array(lib().emu_counts_ptr(self._h), shape=(self.n_samples, 6, lpad))
        return torch.from_numpy(arr)

    def insertions(self):
        k = int(lib().emu_ins_count(self._h))
        nch = int(lib().emu_ins_chars(self._h))
        sample = np.empty(k, np.int32); pos = np.empty(k, np.int32); count = np.empty(k, np.int32)
        off = np.zeros(k + 1, np.int64); chars = np.empty(max(nch, 1), np.uint8)
        lib().emu_ins_export(self._h, _p(sample), _p(pos), _p(count), _p(off), _p(chars))
        raw = chars.tobytes()
        ins = Insertions(sample, pos, count, [raw[int(off[j]):int(off[j + 1])].decode("latin-1") for j in range(k)])
        ins.str_off, ins.chars = off, chars[:int(off[-1])]
        return ins

    def merge_insertions(self, sample, pos, count, str_off, chars):
        chars = np.ascontiguousarray(chars, np.uint8) if len(chars) else np.zeros(1, np.uint8)
        lib().emu_ins_merge(self._h, ctypes.c_longlong(len(pos)), _p(np.ascontiguousarray(sample, np.int32)),
                            _p(np.ascontiguousarray(pos, np.int32)), _p(np.ascontiguousarray(count, np.int32)),
                            _p(np.ascontiguousarray(str_off, np.int64)), _p(chars))

    def call(self, ref_seq, min_depth_consensus=10, min_freq_consensus=0.0, min_depth_variants=1, min_freq_variants=0.03):
        SL = self.n_samples * self.L
        k = max(int(lib().emu_ins_count(self._h)), 1)
        r = CallResult(self.L, self.n_samples, np.empty(SL, np.int32), np.empty(SL, np.int32), np.empty(SL, np.int32),
                       np.empty(SL, np.uint8), np.empty(SL, np.int32), np.empty((SL, 6), np.float64),
                       np.empty((SL, 6), np.int32), np.empty(SL, np.uint8), np.zeros(k, np.float64), np.zeros(k, np.int32),
                       np.zeros(k, np.uint8))
        lib().emu_call(self._h, ctypes.c_char_p(ref_seq.encode("latin-1")), int(min_depth_consensus),
                       ctypes.c_double(min_freq_consensus), int(min_depth_variants), ctypes.c_double(min_freq_variants),
                       _p(r.depth), _p(r.top_id), _p(r.top_count), _p(r.pos_flags), _p(r.ref_count), _p(r.fixed_freq),
                       _p(r.fixed_rank), _p(r.alt_mask), _p(r.ins_freq), _p(r.ins_rank), _p(r.ins_alt))
        return r


def _aligned(a, align=16):
    """16-byte aligned copy that is readable up to the next 16-byte boundary past its end (the staging contract)."""
    buf = np.zeros(a.size + 2 * align, a.dtype)
    o = (-buf.ctypes.data) % align
    v = buf[o:o + a.size]
    v[:] = a
    return v
