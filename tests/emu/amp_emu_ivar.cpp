// amp_emu_ivar.cpp -- TEST INFRASTRUCTURE: the emulator of amp_emu.cpp plus the strand / quality pass and the iVar calling of
// amp_ivar.cuh, the kernels' own source run on the CPU.  Not part of the product.
#include "amp_emu.cpp"
#include "../../amplipy_b200/csrc/amp_ivar.cuh"

#include <cmath>
#include <map>

struct EmuStats {
    std::vector<int> rev; std::vector<unsigned long long> qsum;
    std::vector<int> ins_rev; std::vector<unsigned long long> ins_qsum; std::vector<unsigned char> ins_head;
};
static std::map<void*, EmuStats> g_stats;

extern "C" {

void emu_qstats_enable(void* h) {
    EmuCtx* c = (EmuCtx*)h;
    EmuStats& s = g_stats[h];
    const size_t n = (size_t)c->n_samples * AMP_NCH * c->Lpad;
    s.rev.assign(n, 0); s.qsum.assign(n, 0);
    s.ins_rev.assign(c->slots.size(), 0); s.ins_qsum.assign(c->slots.size(), 0); s.ins_head.assign(c->slots.size(), 0);
}

// amp::cta_qstats over reads [first, first + n), CTA after CTA, as amp_qstats_kernel launches it after the fused kernel; the
// trim outputs (o_*) are the rows the pileup walked when `trimmed`
void emu_qstats_pass(void* h, long long first, long long n, const int32_t* pos, const uint16_t* flag, const int32_t* tlen,
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
    std::vector<int> trev(AMP_NCH * AMP_QS_WT), tq(AMP_NCH * AMP_QS_WT);
    int lo = 0;
    for (long long b = 0; b * AMP_QS_READS < n; ++b) amp::cta_qstats(P, trev.data(), tq.data(), &lo, (int)b, AMP_QS_READS);
}

// amp_qstats_host: one sample's [6][L] sums, the insertion alleles' sums in amp_ins_export order
void emu_qstats_host(void* h, int sample, int32_t* rev, int64_t* qsum, int32_t* ins_rev, int64_t* ins_qsum, uint8_t* ins_head) {
    EmuCtx* c = (EmuCtx*)h;
    EmuStats& s = g_stats.at(h);
    for (int ch = 0; ch < AMP_NCH; ++ch)
        for (int p = 0; p < c->L; ++p) {
            const size_t o = ((size_t)sample * AMP_NCH + ch) * c->Lpad + p;
            rev[(size_t)ch * c->L + p] = s.rev[o]; qsum[(size_t)ch * c->L + p] = (int64_t)s.qsum[o];
        }
    for (unsigned long long k = 0; k < c->cursor[1]; ++k) {
        const unsigned int sl = c->entries[k];
        ins_rev[k] = s.ins_rev[sl]; ins_qsum[k] = (int64_t)s.ins_qsum[sl]; ins_head[k] = s.ins_head[sl];
    }
}

// amp::ivar_position for every (sample, position), on the outputs of emu_call (the serial calling, which links the lists)
void emu_call_ivar(void* h, const char* ref_seq, const int32_t* depth, const int32_t* top_id, const int32_t* top_count,
                   const double* fixed_freq, const int32_t* fixed_rank, const double* ins_freq, const int32_t* ins_rank, int min_depth,
                   double min_freq, double iupac_threshold, uint8_t* iupac, int32_t* fixed_mq, double* fixed_pval, int32_t* ins_mq,
                   double* ins_pval) {
    EmuCtx* c = (EmuCtx*)h;
    EmuStats& s = g_stats.at(h);
    std::vector<int> heads((size_t)c->n_samples * c->Lpad, -1);
    for (unsigned long long k = 0; k < c->cursor[1]; ++k) {   // as emu_call links them
        unsigned int sl = c->entries[k];
        const unsigned char* rec = c->arena.data() + (c->slots[sl].key & 0xFFFFFFFFFFULL) * 8;
        int gpos; memcpy(&gpos, rec, 4);
        c->slots[sl].next = heads[gpos]; heads[gpos] = (int)sl;
    }
    amp::IvarParams P{};
    P.L = c->L; P.Lpad = c->Lpad; P.n_samples = c->n_samples; P.counts = c->counts.data(); P.qsum = s.qsum.data();
    P.slots = c->slots.data(); P.slot_entry = c->slot_entry.data(); P.arena = c->arena.data(); P.heads = heads.data();
    P.ins_qsum = s.ins_qsum.data(); P.ref_seq = (const unsigned char*)ref_seq; P.ref_stride = 0;
    P.depth = depth; P.top_id = top_id; P.top_count = top_count; P.fixed_freq = fixed_freq; P.fixed_rank = fixed_rank;
    P.ins_freq = ins_freq; P.ins_rank = ins_rank;
    P.min_depth = min_depth; P.min_freq = min_freq; P.iupac_threshold = iupac_threshold;
    P.iupac = iupac; P.fixed_mq = fixed_mq; P.fixed_pval = fixed_pval; P.ins_mq = ins_mq; P.ins_pval = ins_pval;
    for (long long gp = 0; gp < (long long)c->n_samples * c->L; ++gp) amp::ivar_position(P, gp);
}

double emu_fisher_less(long long D, long long a, int mq) { return amp::fisher_less(D, a, mq); }

}  // extern "C"
