"""Host-side assembly of the calling kernel's per-position outputs into the reference's products:
the consensus string (AmpliPy.py:919-929, 955-960) and the variant records (AmpliPy.py:932-951).

The arithmetic (depth, float64 frequencies, thresholds, allele order, tie-breaks) is done on the
device by ``amp_call``; this module only walks the flags and formats.
"""
from dataclasses import dataclass
from typing import Dict, List, Tuple

import numpy as np

FIXED_SYMS = "ACGTN-"


@dataclass
class Insertions:
    """Distinct insertion alleles in ``amp_ins_export`` order (dense index k)."""
    sample: np.ndarray      # i32[K]
    pos: np.ndarray         # i32[K]
    count: np.ndarray       # i32[K]
    strs: List[str]         # K python strings

    def as_dict(self, sample=0) -> Dict[Tuple[int, str], int]:
        return {(int(p), s): int(c) for sm, p, c, s in zip(self.sample, self.pos, self.count, self.strs) if sm == sample}

    @property
    def k(self):
        return len(self.strs)


@dataclass
class CallResult:
    """Raw ``amp_call`` outputs for all samples (arrays are [S*L] or [S*L, 6])."""
    L: int
    n_samples: int
    depth: np.ndarray
    top_id: np.ndarray
    top_count: np.ndarray
    pos_flags: np.ndarray
    ref_count: np.ndarray
    fixed_freq: np.ndarray
    fixed_rank: np.ndarray
    alt_mask: np.ndarray
    ins_freq: np.ndarray
    ins_rank: np.ndarray
    ins_alt: np.ndarray


def consensus_string(res: CallResult, ins: Insertions, sample=0, unknown_symbol="N", iupac=None, L=None) -> str:
    """''.join(consensus_symbols) of AmpliPy.py:920-929, 960.  ``iupac``: the IUPAC codes of Engine.call_ivar ([S*L], 0 = keep
    the reference's symbol) replace the symbols of the positions that pass the consensus gate.  ``L``: the sample's own reference
    length when it is shorter than the context's (a contig of a multi-record FASTA)."""
    L = res.L if L is None else L
    sl = slice(sample * res.L, sample * res.L + L)
    top = res.top_id[sl]
    ok = (res.pos_flags[sl] & 1) != 0
    table = np.frombuffer((FIXED_SYMS + unknown_symbol).encode(), np.uint8)
    idx = np.where(ok & (top >= 0) & (top < 6), top, 6)
    chars = table[idx]
    if iupac is not None:
        amb = ok & (iupac[sl] != 0)
        chars = np.where(amb, iupac[sl], chars).astype(np.uint8)
        ok = ok & ~amb
    multi = np.flatnonzero(ok & (top >= 6))
    if multi.size == 0:
        return chars.tobytes().decode()
    out = []
    prev = 0
    raw = chars.tobytes().decode()
    for p in multi:
        out.append(raw[prev:p])
        out.append(ins.strs[int(top[p]) - 6])
        prev = p + 1
    out.append(raw[prev:])
    return "".join(out)


def variant_records(res: CallResult, ins: Insertions, ref_seq: str, counts: np.ndarray, sample=0, L=None):
    """[(pos0, ref, [alts], DP, REF_DP, [ALT_DP], REF_FREQ, [ALT_FREQ], GT tuple)] in reference order
    (AmpliPy.py:932-951): ALT alleles follow the reference's sort (count, freq, symbol descending).
    ``counts`` = this sample's int32[6, L] count matrix (ALT_DP of the fixed symbols); ``L`` as in consensus_string."""
    L = res.L if L is None else L
    base = sample * res.L
    flags = res.pos_flags[base:base + L]
    emit = np.flatnonzero(flags & 2)
    by_pos = {}
    if ins.k:
        sel = np.flatnonzero((ins.sample == sample) & (res.ins_alt[:ins.k] != 0))
        for k, p in zip(sel.tolist(), ins.pos[sel].tolist()):
            by_pos.setdefault(p, []).append(k)
    # the emitting positions' values as plain Python lists (indexing numpy scalars one by one costs more than everything else here)
    ge = emit + base
    fl = flags[emit].tolist()
    masks = res.alt_mask[ge].tolist()
    ranks = res.fixed_rank[ge].tolist()
    freqs = res.fixed_freq[ge].tolist()
    cnts = np.ascontiguousarray(counts[:, emit].T).tolist()
    refc = res.ref_count[ge].tolist()
    depth = res.depth[ge].tolist()
    ins_rank, ins_count, ins_freq = res.ins_rank, ins.count, res.ins_freq
    out = []
    for j, p in enumerate(emit.tolist()):
        alts = []   # (rank, symbol, count, freq)
        m = masks[j]
        if m:
            rk, fq, ct = ranks[j], freqs[j], cnts[j]
            for ch in range(6):
                if m & (1 << ch):
                    alts.append((rk[ch], FIXED_SYMS[ch], ct[ch], fq[ch]))
        for k in by_pos.get(p, ()):
            alts.append((int(ins_rank[k]), ins.strs[k], int(ins_count[k]), float(ins_freq[k])))
        if len(alts) > 1:
            alts.sort(key=lambda a: a[0])
        rc = refc[j]
        ch_ref = FIXED_SYMS.find(ref_seq[p])
        rf = freqs[j][ch_ref] if (rc and ch_ref >= 0) else (rc / depth[j] if rc else 0.0)
        n = len(alts)
        gt = tuple(range(n + 1)) if (fl[j] & 4) else tuple(range(1, n + 1))
        out.append((p, ref_seq[p], [a[1] for a in alts], depth[j], rc, [a[2] for a in alts], rf, [a[3] for a in alts], gt))
    return out
