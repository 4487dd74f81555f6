// amp_exchange.cuh -- the deep-sample exchange of the strand / quality sums (DESIGN.md 5): a rank's insertion table packed with
// each allele's sums into one fixed-size slot, and the merge of the other ranks' slots into every rank's table.  Written as
// __host__ __device__ per-entry bodies so that tests/emu runs this very source on the CPU.
//
//   stats slot = { u64 n_alleles, u64 arena_words,
//                  {u64 arena word offset, u64 count, u64 ins_qsum, u64 ins_rev | ins_head << 32}[cap_entries],
//                  arena bytes [cap_arena] }
//
//   deletion slot = { u64 n_alleles, {u64 key, u64 count, u64 rev, u64 qsum}[cap_entries] }   (the table of amp_dels.cuh)
#pragma once
#include "amp_core.cuh"
#include "amp_dels.cuh"

namespace amp {

#define AMP_XQ_WORDS 4   // u64 words per entry of a stats slot

struct QStatsSlots {                           // the table's per-slot strand / quality sums
    int* ins_rev; unsigned long long* ins_qsum; unsigned char* ins_head;
};

struct ArenaText {   // key characters of a packed record
    const unsigned char* p;
    AMP_HD char operator()(int i) const { return (char)p[i]; }
    AMP_HD uint32_t word(int i, int len) const {
        uint32_t w = *(const uint32_t*)(p + i);                 // records are padded to 8 bytes
        if (len - i < 4) w &= (1u << (8 * (len - i))) - 1u;
        return w;
    }
};

// The table as the pack sees it: n entries and `words` arena words.  cursor[0] runs past the arena when a reservation failed
// (AMP_E_ARENA_FULL); no slot names such a record.  Returns whether it fits the slot.
AMP_HD bool xq_pack_size(const InsTable& T, unsigned long long cap_entries, unsigned long long cap_arena_words, unsigned long long& n,
                         unsigned long long& words) {
    words = T.cursor[0] < T.arena_words ? T.cursor[0] : T.arena_words;
    n = T.cursor[1];
    return n <= cap_entries && words <= cap_arena_words;
}
// The slot's two header words, by one thread.  A table that does not fit packs as empty and sets the error bit.
AMP_HD void xq_pack_header(const InsTable& T, unsigned long long* slot, bool fits, unsigned long long n, unsigned long long words,
                           unsigned long long cap_entries) {
    slot[0] = fits ? n : 0ULL; slot[1] = fits ? words : 0ULL;
    if (!fits) atomic_or(T.err, n > cap_entries ? AMP_E_TABLE_FULL : AMP_E_ARENA_FULL);
}
// Entry k of the slot: allele k of the table with its sums.
AMP_HD void xq_pack_entry(const InsTable& T, const QStatsSlots& Q, unsigned long long* slot, unsigned long long k) {
    const unsigned int s = T.entries[k];
    unsigned long long* e = slot + 2 + AMP_XQ_WORDS * k;
    e[0] = T.slots[s].key & 0xFFFFFFFFFFULL;
    e[1] = (unsigned long long)(unsigned int)T.slots[s].count;
    e[2] = Q.ins_qsum[s];
    e[3] = (unsigned long long)(unsigned int)Q.ins_rev[s] | ((unsigned long long)Q.ins_head[s] << 32);
}
AMP_HD unsigned long long* xq_slot_arena(unsigned long long* slot, unsigned long long cap_entries) { return slot + 2 + AMP_XQ_WORDS * cap_entries; }

// One allele of another rank added to this rank's table with its sums.  A known allele takes the count and the sums in its own
// slot.  A new one is added by ins_table_add, as the plain merge adds it, and its sums go to the slot it was given; an allele that
// could not be placed (AMP_E_TABLE_FULL / AMP_E_ARENA_FULL, whose bit reports the loss) gets no sums.
template <class Text>
AMP_HD void ins_merge_qstats(const InsTable& T, const QStatsSlots& Q, int gpos, int len, const Text& t, int count, int rev,
                             unsigned long long qsum, bool head) {
    int s = ins_table_find(T, gpos, len, t);
    if (s >= 0) {
        atomic_add(&T.slots[s].count, count);
    } else {
        ins_table_add(T, gpos, len, t, count);
        s = ins_table_find(T, gpos, len, t);
        if (s < 0) return;
    }
    if (rev) atomic_add(&Q.ins_rev[s], rev);
    if (qsum) atomic_add64(&Q.ins_qsum[s], qsum);
    if (head) Q.ins_head[s] = 1;
}
// Entry k of another rank's slot merged into this rank's table.
AMP_HD void xq_merge_entry(const InsTable& T, const QStatsSlots& Q, const unsigned long long* slot, unsigned long long cap_entries,
                           unsigned long long k) {
    const unsigned long long* e = slot + 2 + AMP_XQ_WORDS * k;
    const unsigned char* rec = (const unsigned char*)(slot + 2 + AMP_XQ_WORDS * cap_entries) + e[0] * 8;
    const int gpos = ((const int*)rec)[0];
    const int len = (int)((const unsigned int*)rec)[1];
    ArenaText t{rec + 8};
    ins_merge_qstats(T, Q, gpos, len, t, (int)e[1], (int)(unsigned int)e[3], e[2], (e[3] >> 32) != 0);
}

#define AMP_XD_WORDS 4   // u64 words per entry of a deletion slot

// The deletion table as the pack sees it: n alleles.  Returns whether they fit the slot.
AMP_HD bool xd_pack_size(const DelTable& T, unsigned long long cap_entries, unsigned long long& n) {
    n = T.cursor[0];
    return n <= cap_entries;
}
// The slot's header word, by one thread.  A table that does not fit packs as empty and sets AMP_E_DELS_FULL.
AMP_HD void xd_pack_header(const DelTable& T, unsigned long long* slot, bool fits, unsigned long long n) {
    slot[0] = fits ? n : 0ULL;
    if (!fits) atomic_or(T.err, AMP_E_DELS_FULL);
}
// Entry k of the slot: allele k of the table with its sums.
AMP_HD void xd_pack_entry(const DelTable& T, unsigned long long* slot, unsigned long long k) {
    const DelSlot& s = T.slots[T.entries[k]];
    unsigned long long* e = slot + 1 + AMP_XD_WORDS * k;
    e[0] = s.key; e[1] = s.cr & 0xFFFFFFFFULL; e[2] = s.cr >> 32; e[3] = s.qsum;
}
// Entry k of another rank's slot added to this rank's table.
AMP_HD void xd_merge_entry(const DelTable& T, const unsigned long long* slot, unsigned long long k) {
    const unsigned long long* e = slot + 1 + AMP_XD_WORDS * k;
    del_table_add(T, (int)(e[0] >> 32), (int)(e[0] & 0xFFFFFFFFu), (unsigned int)e[1], (unsigned int)e[2], e[3]);
}

}  // namespace amp
