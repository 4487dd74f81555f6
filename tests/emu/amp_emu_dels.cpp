// amp_emu_dels.cpp -- TEST INFRASTRUCTURE: the emulator of amp_emu_dist.cpp plus the anchored deletion alleles (amp_dels.cuh): the
// strand / quality pass with the table (cta_qstats<true>), their calling (amp_ivar.cuh ivar_del) and their deep-sample pack / merge
// (amp_exchange.cuh), the kernels' own source run on the CPU.  Not part of the product.
#include "amp_emu_dist.cpp"

#include <algorithm>

struct EmuDels {
    std::vector<amp::DelSlot> slots; std::vector<unsigned int> entries; unsigned long long cursor = 0;
};
static std::map<void*, EmuDels> g_dels;

static amp::DelTable emu_dels_table(void* h) {
    EmuDels& d = g_dels.at(h);
    return amp::DelTable{d.slots.data(), d.slots.size() - 1, d.entries.data(), &d.cursor, &((EmuCtx*)h)->err};
}

// list positions sorted by key: the order of amp_dels_export
static std::vector<unsigned long long> emu_dels_order(void* h) {
    EmuDels& d = g_dels.at(h);
    std::vector<unsigned long long> o(d.cursor);
    for (unsigned long long k = 0; k < d.cursor; ++k) o[k] = k;
    std::sort(o.begin(), o.end(), [&](unsigned long long a, unsigned long long b) { return d.slots[d.entries[a]].key < d.slots[d.entries[b]].key; });
    return o;
}

extern "C" {

// amp_dels_enable: `slots` a power of two
void emu_dels_enable(void* h, long long slots) {
    EmuDels& d = g_dels[h];
    d.slots.assign((size_t)slots, amp::DelSlot{0, 0, 0});
    d.entries.assign((size_t)slots, 0);
    d.cursor = 0;
}

// amp_dels_reset_kernel: the listed slots, then the cursor (emu_reset clears the error word)
void emu_dels_reset(void* h) {
    EmuDels& d = g_dels.at(h);
    for (unsigned long long k = 0; k < d.cursor; ++k) d.slots[d.entries[k]] = amp::DelSlot{0, 0, 0};
    d.cursor = 0;
}

// emu_qstats_pass with the table: amp_qstats_dels_kernel
void emu_qstats_dels_pass(void* h, long long first, long long n, const int32_t* pos, const uint16_t* flag, const int32_t* tlen,
                          const uint32_t* cig_off, const uint32_t* cigar, const uint32_t* seq_off, const uint8_t* seq,
                          const uint32_t* qual_off, const uint8_t* qual, int trimmed, int sample, int32_t* o_pos, uint16_t* o_ncig,
                          uint8_t* o_flags, uint32_t* o_cigar) {
    EmuCtx* c = (EmuCtx*)h;
    EmuStats& s = g_stats.at(h);
    amp::QStatsParams P{};
    P.b = amp::BatchPtrs{first, n, pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual};
    P.o = amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar};
    P.trimmed = trimmed; P.L = c->L; P.Lpad = c->Lpad; P.minq = c->tp.min_quality; P.gpos_base = sample * c->Lpad;
    P.rev = s.rev.data() + (size_t)sample * AMP_NCH * c->Lpad; P.qsum = s.qsum.data() + (size_t)sample * AMP_NCH * c->Lpad;
    P.tab = c->tab; P.ins_rev = s.ins_rev.data(); P.ins_qsum = s.ins_qsum.data(); P.ins_head = s.ins_head.data(); P.err = &c->err;
    P.dels = emu_dels_table(h);
    std::vector<int> trev(AMP_NCH * AMP_QS_WT), tq(AMP_NCH * AMP_QS_WT);
    int lo = 0;
    for (long long b = 0; b * AMP_QS_READS < n; ++b) amp::cta_qstats<true>(P, trev.data(), tq.data(), &lo, (int)b, AMP_QS_READS);
}

long long emu_dels_count(void* h) { return (long long)g_dels.at(h).cursor; }

// amp_dels_export
void emu_dels_export(void* h, int32_t* sample, int32_t* anchor, int32_t* len, int32_t* count, int32_t* rev, int64_t* qsum) {
    EmuDels& d = g_dels.at(h);
    const std::vector<unsigned long long> o = emu_dels_order(h);
    for (size_t j = 0; j < o.size(); ++j) {
        const amp::DelSlot& s = d.slots[d.entries[o[j]]];
        amp::del_key_split(s.key, ((EmuCtx*)h)->Lpad, sample[j], anchor[j], len[j]);
        count[j] = (int32_t)(s.cr & 0xFFFFFFFFULL); rev[j] = (int32_t)(s.cr >> 32); qsum[j] = (int64_t)s.qsum;
    }
}

// amp_dels_merge_kernel
void emu_dels_merge(void* h, long long n, const int32_t* sample, const int32_t* anchor, const int32_t* len, const int32_t* count,
                    const int32_t* rev, const int64_t* qsum) {
    const amp::DelTable T = emu_dels_table(h);
    const int lpad = ((EmuCtx*)h)->Lpad;
    for (long long k = 0; k < n; ++k)
        amp::del_table_add(T, sample[k] * lpad + anchor[k], len[k], (unsigned)count[k], (unsigned)rev[k], (unsigned long long)qsum[k]);
}

// amp_ivar_dels_kernel on the depths of emu_call, outputs in export order
void emu_call_ivar_dels(void* h, const int32_t* depth, int min_depth, double min_freq, int32_t* mq, double* pval) {
    EmuCtx* c = (EmuCtx*)h;
    const unsigned long long n = g_dels.at(h).cursor;
    std::vector<int> m(n); std::vector<double> pv(n);
    amp::IvarDelParams P{};
    P.L = c->L; P.Lpad = c->Lpad; P.dels = emu_dels_table(h); P.n = n; P.depth = depth; P.min_depth = min_depth; P.min_freq = min_freq;
    P.mq = m.data(); P.pval = pv.data();
    for (unsigned long long k = 0; k < n; ++k) amp::ivar_del(P, k);
    const std::vector<unsigned long long> o = emu_dels_order(h);
    for (size_t j = 0; j < o.size(); ++j) { mq[j] = m[o[j]]; pval[j] = pv[o[j]]; }
}

// amp_dels_pack_kernel as one thread
void emu_dels_pack(void* h, unsigned long long* slot, long long cap_entries) {
    const amp::DelTable T = emu_dels_table(h);
    unsigned long long n;
    const bool fits = amp::xd_pack_size(T, (unsigned long long)cap_entries, n);
    amp::xd_pack_header(T, slot, fits, n);
    if (!fits) return;
    for (unsigned long long k = 0; k < n; ++k) amp::xd_pack_entry(T, slot, k);
}

// amp_dels_merge_packed_kernel, rank after rank
void emu_dels_merge_packed(void* h, const unsigned long long* slots, int n_ranks, int my_rank, long long cap_entries) {
    const amp::DelTable T = emu_dels_table(h);
    const unsigned long long slot_words = 1 + AMP_XD_WORDS * (unsigned long long)cap_entries;
    for (int r = 0; r < n_ranks; ++r) {
        if (r == my_rank) continue;
        const unsigned long long* slot = slots + (unsigned long long)r * slot_words;
        for (unsigned long long k = 0; k < slot[0]; ++k) amp::xd_merge_entry(T, slot, k);
    }
}

// the home slot of a key (tests choose colliding keys with it)
unsigned long long emu_dels_home(int gpos, int len, long long slots) { return amp::mix64(amp::del_key(gpos, len)) & (unsigned long long)(slots - 1); }

}  // extern "C"
