"""The step around the fused kernel: insertion alleles are linked into their position's list where they are created
(amp::ins_table_add) and one kernel resets the context.  The lists have to be current after every launch that adds
alleles, and a reset has to leave nothing behind.  The calling kernel's body (amp_call.cuh) runs on the CPU emulation too."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import emu_driver
import golden_io
import parity
from amplipy_b200 import synth
from amplipy_b200.calling import CallResult
from amplipy_b200.primers import find_overlapping_primers, max_primer_len

FIELDS = ["depth", "top_id", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask", "ins_freq",
          "ins_rank", "ins_alt"]
POS_FIELDS = ["depth", "top_count", "pos_flags", "ref_count", "fixed_freq", "fixed_rank", "alt_mask"]


def _bitwise_equal(a, b, fields=FIELDS):
    return [f for f in fields if np.ascontiguousarray(getattr(a, f)).tobytes() != np.ascontiguousarray(getattr(b, f)).tobytes()]


# ---------------------------------------------------------------------------------------------------------------- CPU
_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "amplipy_b200", "csrc")


@pytest.fixture(scope="module")
def call_emu():
    """tests/emu/amp_emu_call.cpp built into a library of its own (the whole emulator plus the calling kernel's body),
    with the restypes emu_driver.lib() sets."""
    so = os.path.join(_HERE, "emu", "libamp_emu_call.so")
    srcs = [os.path.join(_HERE, "emu", f) for f in ("amp_emu_call.cpp", "amp_emu.cpp")] + \
        [os.path.join(_CSRC, f) for f in ("amp_core.cuh", "amp_kernels.cuh", "amp_warp.cuh", "amp_call.cuh", "amp_bgzf.cuh", "amp_ont.cuh",
                                          "amp_deflate.cuh")]
    if not os.path.isfile(so) or any(os.path.getmtime(f) > os.path.getmtime(so) for f in srcs):
        gxx = "/usr/bin/g++" if os.path.isfile("/usr/bin/g++") else "g++"
        subprocess.check_call([gxx, "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-variable", "-Wno-unused-function", "-O2",
                               "-o", so, srcs[0]])
    lib = ctypes.CDLL(so)
    lib.emu_create.restype = ctypes.c_void_p
    lib.emu_ins_count.restype = ctypes.c_longlong
    lib.emu_ins_chars.restype = ctypes.c_longlong
    lib.emu_error_flags.restype = ctypes.c_uint
    return lib


def _engine_with_lists(lib, monkeypatch, **kw):
    monkeypatch.setattr(emu_driver, "lib", lambda: lib)
    eng = emu_driver.EmuEngine(**kw)
    lib.emu_keep_lists(eng._h)
    return eng


def _call_kernel(lib, eng, ref_seq, mdc, mfc, mdv, mfv):
    """emu_driver.EmuEngine.call with the kernel's body in place of the serial form."""
    SL = eng.n_samples * eng.L
    k = max(int(lib.emu_ins_count(eng._h)), 1)
    r = CallResult(eng.L, eng.n_samples, np.empty(SL, np.int32), np.empty(SL, np.int32), np.empty(SL, np.int32),
                   np.empty(SL, np.uint8), np.empty(SL, np.int32), np.empty((SL, 6), np.float64), np.empty((SL, 6), np.int32),
                   np.empty(SL, np.uint8), np.zeros(k, np.float64), np.zeros(k, np.int32), np.zeros(k, np.uint8))
    p = emu_driver._p
    lib.emu_call_kernel(eng._h, ctypes.c_char_p(ref_seq.encode("latin-1")), int(mdc), ctypes.c_double(mfc), int(mdv),
                        ctypes.c_double(mfv), p(r.depth), p(r.top_id), p(r.top_count), p(r.pos_flags), p(r.ref_count),
                        p(r.fixed_freq), p(r.fixed_rank), p(r.alt_mask), p(r.ins_freq), p(r.ins_rank), p(r.ins_alt))
    return r


@pytest.mark.parametrize("name", golden_io.list_cases())
def test_emulated_kernel_body_matches_serial_calling(name, call_emu, monkeypatch):
    """Lists linked by ins_table_add as the alleles are created, then amp::call_thread on the fiber runtime against the
    serial amp::call_position (which links its own lists): every output bit for bit, long allele lists (cfg4_ont*) and
    quirks included."""
    b, meta, arr = golden_io.load_case(name)
    p = meta["params"]
    eng = _engine_with_lists(call_emu, monkeypatch, **parity.engine_kwargs(meta))
    eng.process(b, trim=True, pileup=True)
    args = (bytes(arr["ref_seq"]).decode(), p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"],
            p["min_freq_variants"])
    got = _call_kernel(call_emu, eng, *args)
    want = eng.call(*args)
    call_emu.emu_destroy(eng._h)
    eng._h = None
    assert _bitwise_equal(got, want) == []


def test_emulated_plate_same_position_alleles(call_emu, monkeypatch):
    """Three samples, alleles at the same positions in samples 0 and 2 (sample 1 empty): lists are per (sample, position)."""
    b, meta, arr = golden_io.load_case("fuzz1")
    p = meta["params"]
    eng = _engine_with_lists(call_emu, monkeypatch, n_samples=3, **parity.engine_kwargs(meta))
    eng.process(b, trim=True, pileup=True, sample=0)
    eng.process(b, trim=True, pileup=True, sample=2, first=0, n=b.n // 2)
    args = (bytes(arr["ref_seq"]).decode(), p["min_depth_consensus"], p["min_freq_consensus"], p["min_depth_variants"],
            p["min_freq_variants"])
    ins = eng.insertions()
    assert set(ins.sample.tolist()) == {0, 2}
    assert set(ins.pos[ins.sample == 0].tolist()) & set(ins.pos[ins.sample == 2].tolist())
    got = _call_kernel(call_emu, eng, *args)
    want = eng.call(*args)
    call_emu.emu_destroy(eng._h)
    eng._h = None
    assert _bitwise_equal(got, want) == []


# ---------------------------------------------------------------------------------------------------------------- GPU
L = 29903


@pytest.fixture(scope="module")
def workload():
    g = synth.random_genome(L, 11)
    primers, amps = synth.make_scheme(L, 98, seed=3)
    prim = [(s, e) for s, e, _ in primers]
    return dict(g=g, amps=amps, prim=prim, tables=find_overlapping_primers(L, prim, 0), mpl=max_primer_len(prim))


def _engine(w, **kw):
    from amplipy_b200.engine import Engine
    return Engine(ref_len=L, primer_tables=w["tables"], max_primer_len=w["mpl"], device=0, **kw)


def _canonical(res, ins, n_samples=1):
    """Calling outputs with the insertion alleles named by (sample, position, string) instead of their dense index, whose
    order depends on the order in which alleles were first seen."""
    key = [(int(ins.sample[k]), int(ins.pos[k]), ins.strs[k]) for k in range(ins.k)]
    top = [int(t) if t < 6 else key[t - 6] for t in res.top_id.tolist()]
    per_allele = {key[k]: (float(res.ins_freq[k]).hex(), int(res.ins_rank[k]), int(res.ins_alt[k])) for k in range(ins.k)}
    return {f: np.ascontiguousarray(getattr(res, f)).tobytes() for f in POS_FIELDS}, top, per_allele


@pytest.mark.gpu
def test_call_twice_without_reset(workload):
    w = workload
    eng = _engine(w)
    eng.process(synth.ont_batch(w["g"], w["amps"], 3_000, seed=21), trim=True, pileup=True)
    r1 = eng.call(w["g"])
    r2 = eng.call(w["g"])
    assert eng.error_flags() == 0
    assert _bitwise_equal(r1, r2) == []
    eng.close()


@pytest.mark.gpu
def test_call_between_batches(workload):
    """process A, call, process B, call == process A + B, call: the lists grow with every launch."""
    w = workload
    b = synth.illumina_batch(w["g"], w["amps"], 40_000, seed=22, p_ins=0.05)
    h = b.n // 2
    split = _engine(w)
    split.process(b.slice(0, h), trim=True, pileup=True)
    split.call(w["g"])
    split.process(b.slice(h, b.n), trim=True, pileup=True)
    got = _canonical(split.call(w["g"]), split.insertions())
    whole = _engine(w)
    whole.process(b, trim=True, pileup=True)
    want = _canonical(whole.call(w["g"]), whole.insertions())
    assert split.error_flags() == 0 and whole.error_flags() == 0
    assert got == want
    split.close(); whole.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["reset_async", "reset"])
def test_reset_leaves_no_alleles(workload, how):
    """An indel-rich batch (thousands of alleles), a reset, then a batch without insertions: no insertion outputs, no
    top allele that is an insertion, and calling equal to that of a fresh context."""
    import torch
    w = workload
    clean = synth.illumina_batch(w["g"], w["amps"], 20_000, seed=23, p_ins=0.0)
    eng = _engine(w)
    eng.process(synth.ont_batch(w["g"], w["amps"], 3_000, seed=24), trim=True, pileup=True)
    eng.call(w["g"])
    assert eng.insertions().k > 1000
    if how == "reset_async":
        s = torch.cuda.Stream()
        eng.reset_async(s.cuda_stream)
        s.synchronize()
    else:
        eng.reset()
    assert eng.insertions().k == 0 and eng.error_flags() == 0
    eng.process(clean, trim=True, pileup=True)
    res = eng.call(w["g"])
    assert eng.insertions().k == 0
    assert res.top_id.max() < 6
    fresh = _engine(w)
    fresh.process(clean, trim=True, pileup=True)
    assert _bitwise_equal(res, fresh.call(w["g"])) == []
    eng.close(); fresh.close()


@pytest.mark.gpu
def test_merged_alleles_are_called(workload):
    """Alleles added by amp_ins_merge (host) and amp_ins_merge_packed (device) join the lists like the kernel's own."""
    import torch
    w = workload
    b = synth.ont_batch(w["g"], w["amps"], 3_000, seed=25)
    src = _engine(w)
    src.process(b, trim=True, pileup=True)
    ins = src.insertions()
    counts = src.counts()
    want = _canonical(src.call(w["g"]), ins)
    # host merge into a context holding the same counts
    dst = _engine(w)
    dst.upload_counts(counts)
    dst.merge_insertions(ins.sample, ins.pos, ins.count, ins.str_off, ins.chars)
    assert _canonical(dst.call(w["g"]), dst.insertions()) == want
    # device merge: rank 0's packed table merged into rank 1's empty one
    cap_e, cap_a = 1 << 18, 1 << 24
    buf = torch.zeros(2 * src.ins_slot_bytes(cap_e, cap_a) // 8, dtype=torch.int64, device="cuda")
    src.ins_pack_device(buf.data_ptr(), cap_e, cap_a)
    torch.cuda.synchronize()
    dev = _engine(w)
    dev.upload_counts(counts)
    dev.ins_merge_packed(buf.data_ptr(), 2, 1, cap_e, cap_a)
    torch.cuda.synchronize()
    assert dev.error_flags() == 0
    assert _canonical(dev.call(w["g"]), dev.insertions()) == want
    src.close(); dst.close(); dev.close()


@pytest.mark.gpu
def test_plate_same_position_alleles(workload):
    """A few-sample plate with insertion alleles at the same positions in different samples: each sample's calling equals
    that of a context of its own."""
    w = workload
    batches = [synth.illumina_batch(w["g"], w["amps"], 20_000, seed=30 + s, p_ins=0.05) for s in range(3)]
    plate = _engine(w, n_samples=4)
    for s, b in enumerate(batches):
        plate.process(b, trim=True, pileup=True, sample=s if s < 2 else 3)
    res = plate.call(w["g"])
    ins = plate.insertions()
    assert len(set(ins.pos[ins.sample == 0].tolist()) & set(ins.pos[ins.sample == 3].tolist())) > 10
    assert plate.error_flags() == 0
    for s, b in enumerate(batches):
        ps = s if s < 2 else 3
        one = _engine(w)
        one.process(b, trim=True, pileup=True)
        r1, i1 = one.call(w["g"]), one.insertions()
        rows = slice(ps * L, (ps + 1) * L)
        for f in POS_FIELDS:
            assert np.array_equal(getattr(res, f)[rows], getattr(r1, f)), (s, f)
        assert np.array_equal(res.fixed_freq[rows].view(np.int64), r1.fixed_freq.view(np.int64))
        mine = np.flatnonzero(ins.sample == ps)
        got = {(int(ins.pos[k]), ins.strs[k]): (float(res.ins_freq[k]).hex(), int(res.ins_rank[k]), int(res.ins_alt[k])) for k in mine}
        want = {(int(i1.pos[k]), i1.strs[k]): (float(r1.ins_freq[k]).hex(), int(r1.ins_rank[k]), int(r1.ins_alt[k])) for k in range(i1.k)}
        assert got == want
        one.close()
    plate.close()
