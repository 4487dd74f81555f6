// amp_emu_dist.cpp -- TEST INFRASTRUCTURE: the emulator of amp_emu_ivar.cpp plus the deep-sample exchange of the strand / quality
// sums (amp_exchange.cuh), the kernels' own per-entry bodies run on the CPU.  Not part of the product.
#include "amp_emu_ivar.cpp"
#include "../../amplipy_b200/csrc/amp_exchange.cuh"

extern "C" {

// the [n_samples][6][Lpad] sums the strand / quality pass accumulates into (the all-reduce of the host form works on them in place)
int* emu_rev_ptr(void* h) { return g_stats.at(h).rev.data(); }
unsigned long long* emu_qsum_ptr(void* h) { return g_stats.at(h).qsum.data(); }

static amp::QStatsSlots emu_qslots(void* h) {
    EmuStats& s = g_stats.at(h);
    return amp::QStatsSlots{s.ins_rev.data(), s.ins_qsum.data(), s.ins_head.data()};
}

// emu_ins_merge with each allele's sums (amp_exchange.cuh ins_merge_qstats): the host form of the exchange
void emu_ins_merge_qstats(void* h, long long n, const int32_t* sample, const int32_t* pos, const int32_t* count, const int64_t* str_off,
                          const char* chars, const int32_t* ins_rev, const int64_t* ins_qsum, const uint8_t* ins_head) {
    EmuCtx* c = (EmuCtx*)h;
    const amp::QStatsSlots q = emu_qslots(h);
    for (long long k = 0; k < n; ++k) {
        RawText t{chars + str_off[k]};
        amp::ins_merge_qstats(c->tab, q, sample[k] * c->Lpad + pos[k], (int)(str_off[k + 1] - str_off[k]), t, count[k], ins_rev[k],
                              (unsigned long long)ins_qsum[k], ins_head[k] != 0);
    }
}

// amp_ins_pack_qstats_kernel as one thread: the table with its sums -> one stats slot
void emu_ins_pack_qstats(void* h, unsigned long long* slot, long long cap_entries, long long cap_arena_bytes) {
    EmuCtx* c = (EmuCtx*)h;
    const amp::QStatsSlots q = emu_qslots(h);
    unsigned long long n, words;
    const bool fits = amp::xq_pack_size(c->tab, (unsigned long long)cap_entries, (unsigned long long)(cap_arena_bytes + 7) / 8, n, words);
    amp::xq_pack_header(c->tab, slot, fits, n, words, (unsigned long long)cap_entries);
    if (!fits) return;
    for (unsigned long long k = 0; k < n; ++k) amp::xq_pack_entry(c->tab, q, slot, k);
    memcpy(amp::xq_slot_arena(slot, (unsigned long long)cap_entries), c->arena.data(), words * 8);
}

// amp_ins_merge_packed_qstats_kernel, rank after rank: every slot but my_rank's merged into the table
void emu_ins_merge_packed_qstats(void* h, const unsigned long long* slots, int n_ranks, int my_rank, long long cap_entries,
                                 long long cap_arena_bytes) {
    EmuCtx* c = (EmuCtx*)h;
    const amp::QStatsSlots q = emu_qslots(h);
    const unsigned long long slot_words = 2 + AMP_XQ_WORDS * (unsigned long long)cap_entries + (unsigned long long)(cap_arena_bytes + 7) / 8;
    for (int r = 0; r < n_ranks; ++r) {
        if (r == my_rank) continue;
        const unsigned long long* slot = slots + (unsigned long long)r * slot_words;
        for (unsigned long long k = 0; k < slot[0]; ++k) amp::xq_merge_entry(c->tab, q, slot, (unsigned long long)cap_entries, k);
    }
}

}  // extern "C"
