// amp_dels.cuh -- the anchored deletion alleles of the iVar TSV (DESIGN.md 3.7, --ivar_deletions): a fixed-key open-addressing
// hash table in HBM, filled by the strand / quality pass (amp_ivar.cuh), and its deep-sample pack / merge (amp_exchange.cuh).
// Written as __host__ __device__ code so that tests/emu runs this very source on the CPU.
//
// An allele is (sample, anchor position a, length n): a D op of n bases that directly follows an M / = / X op, whose last base
// (the anchor, at a) passed the quality gate.  Its key is gpos << 32 | n with gpos = sample * Lpad + a; n >= 1, so no key is 0,
// the value of a free slot.  A slot is claimed by CAS on its key; the sums are added atomically, so any read order and any
// partition of the reads over ranks give the same table.  The claimed slots are listed densely (export, reset, pack).
#pragma once
#include "amp_core.cuh"

#define AMP_E_DELS_FULL 128  // anchored deletion table full (amp_dels_enable)

namespace amp {

struct DelSlot {
    unsigned long long key;     // 0 = free
    unsigned long long cr;      // count | rev << 32: one atomic per event for both
    unsigned long long qsum;    // anchor qualities
};

struct DelTable {
    DelSlot* slots; unsigned long long mask;    // capacity - 1 (power of two); slots == nullptr: no table
    unsigned int* entries;                      // entries[k] = slot of the k-th distinct allele
    unsigned long long* cursor;                 // [0] = entries used
    unsigned int* err;
};

AMP_HD unsigned long long del_key(int gpos, int len) { return ((unsigned long long)(unsigned int)gpos << 32) | (unsigned int)len; }

// Add `count` events (`rev` of them from reverse-strand reads, anchor qualities summing to `qsum`) to allele (gpos, len).
AMP_HD void del_table_add(const DelTable& T, int gpos, int len, unsigned int count, unsigned int rev, unsigned long long qsum) {
    const unsigned long long key = del_key(gpos, len);
    unsigned long long slot = mix64(key) & T.mask;
    for (unsigned long long probes = 0; probes <= T.mask; ++probes, slot = (slot + 1) & T.mask) {
        unsigned long long k = ld_cg64(&T.slots[slot].key);
        if (k == 0) {
            k = atomic_cas64(&T.slots[slot].key, 0ULL, key);
            if (k == 0) {
                const unsigned long long e = atomic_add64(T.cursor, 1ULL);
                T.entries[e] = (unsigned int)slot;
                k = key;
            }
        }
        if (k == key) {
            atomic_add64(&T.slots[slot].cr, (unsigned long long)count | ((unsigned long long)rev << 32));
            if (qsum) atomic_add64(&T.slots[slot].qsum, qsum);
            return;
        }
    }
    atomic_or(T.err, AMP_E_DELS_FULL);
}

// Sample, anchor, length of a key (lpad: the context's row stride)
AMP_HD void del_key_split(unsigned long long key, int lpad, int& sample, int& anchor, int& len) {
    const int gpos = (int)(key >> 32);
    sample = gpos / lpad; anchor = gpos - sample * lpad; len = (int)(key & 0xFFFFFFFFu);
}

}  // namespace amp
