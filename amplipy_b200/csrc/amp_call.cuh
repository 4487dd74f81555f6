// amp_call.cuh -- the calling kernel's body (AmpliPy.py:756-771, 919-951), written against warp primitives that are the
// hardware's on the device and the fiber runtime's in tests/emu, so that the CPU emulation runs this very source and checks
// it against the serial form amp::call_position.
//
// Sixteen lanes per (sample, position), one allele per lane (call_group).  A lane per position for the positions without
// insertion alleles, with the groups kept for the others, measured slower on short-read data: a quarter of the
// positions of config 2 carry alleles, and a warp then works through several groups' dependent list walks one after the
// other (DESIGN.md 3.3).
#pragma once
#include "amp_warp.cuh"

namespace amp {

// collectives of the lanes in mask m (a group of sixteen, or the warp)
#if defined(__CUDA_ARCH__)
AMP_WD int g_shfl(unsigned m, int v, int src) { return __shfl_sync(m, v, src); }
AMP_WD double g_shfl(unsigned m, double v, int src) { return __shfl_sync(m, v, src); }
AMP_WD const unsigned char* g_shfl(unsigned m, const unsigned char* v, int src) {
    return (const unsigned char*)__shfl_sync(m, (unsigned long long)v, src);
}
AMP_WD int g_shfl_xor(unsigned m, int v, int d) { return __shfl_xor_sync(m, v, d); }
AMP_WD double g_shfl_xor(unsigned m, double v, int d) { return __shfl_xor_sync(m, v, d); }
AMP_WD unsigned g_ballot(unsigned m, bool p) { return __ballot_sync(m, p); }
AMP_WD int ffs32(unsigned x) { return __ffs((int)x); }
AMP_WD int clz32(unsigned x) { return __clz((int)x); }
#else
// The fiber runtime's collectives span the warp.  Both groups of a warp reach their k-th collective together and a
// lane only reads lanes of its own group, so group-divergent code exchanges the right values; 64-bit values take two
// exchanges.
AMP_WD int g_shfl(unsigned, int v, int src) { return w_shfl(v, src); }
AMP_WD unsigned long long g_shfl_u64(unsigned long long v, int src) {
    const unsigned lo = (unsigned)w_shfl((int)(unsigned)v, src), hi = (unsigned)w_shfl((int)(unsigned)(v >> 32), src);
    return ((unsigned long long)hi << 32) | lo;
}
AMP_WD double g_shfl(unsigned, double v, int src) {
    unsigned long long u; memcpy(&u, &v, 8); u = g_shfl_u64(u, src); memcpy(&v, &u, 8); return v;
}
AMP_WD const unsigned char* g_shfl(unsigned, const unsigned char* v, int src) {
    return (const unsigned char*)(uintptr_t)g_shfl_u64((unsigned long long)(uintptr_t)v, src);
}
AMP_WD int g_shfl_xor(unsigned m, int v, int d) { return g_shfl(m, v, (c_tid() & 31) ^ d); }
AMP_WD double g_shfl_xor(unsigned m, double v, int d) { return g_shfl(m, v, (c_tid() & 31) ^ d); }
AMP_WD unsigned g_ballot(unsigned m, bool p) { return w_ballot(p) & m; }
AMP_WD int ffs32(unsigned x) { return __builtin_ffs((int)x); }
AMP_WD int clz32(unsigned x) { return x ? __builtin_clz(x) : 32; }
#endif

#define AMP_CALL_LANES 16

AMP_HD bool ins_slot_greater(const CallParams& P, int t, int ct, int c, const Sym& me) {
    return ct > c || (ct == c && sym_cmp(slot_sym(P, t), me) > 0);
}

// Positions with more than ten insertion alleles (indel-rich data: every position of an ONT-like sample): the same
// results as amp::call_position, with the sixteen lanes of the group sharing the allele list -- lane l owns entries
// l, l + 16, ... and, for each, walks the whole list once to find its place in the reference's order; the fixed
// symbols are owned by lanes 0..5.  All lanes walk the same addresses in the same order, so the loads are broadcasts.
AMP_WD_COLD void call_long_list(const CallParams& P, const unsigned char* fixed_syms, long long gp, int sample, int p, int ch, int g0,
                                unsigned gmask) {
    constexpr int G = AMP_CALL_LANES;
    const int* cnt = P.counts + (size_t)sample * AMP_NCH * P.Lpad;
    const int head = P.heads[(size_t)sample * P.Lpad + p];
    int cfix[AMP_NCH]; long long total = 0;
AMP_UNROLL
    for (int o = 0; o < AMP_NCH; ++o) { cfix[o] = cnt[(size_t)o * P.Lpad + p]; total += cfix[o]; }
    for (int t = head; t >= 0;) { const InsSlot sl = P.slots[t]; total += sl.count; t = sl.next; }
    const unsigned char refsym = P.ref_seq[(size_t)sample * (size_t)P.ref_stride + p];
    int n_alt = 0, alt_fixed = 0;
    int top_id = -1, top_c = 0;                 // set by the lane that owns the first allele of the order
    int ref_key = -1, refc = 0; double reff = 0.0;   // 936-937: the last match in visiting order wins
    if (ch < AMP_NCH) {
        const int c = cnt[(size_t)ch * P.Lpad + p];          // (cfix[ch] would put the array in local memory)
        const double f = total ? (double)c / (double)total : 0.0;
        int rank = -1;
        if (c) {
            Sym me; me.p = fixed_syms + ch; me.len = 1;
            rank = 0;
AMP_UNROLL
            for (int o = 0; o < AMP_NCH; ++o)
                if (o != ch && cfix[o]) { Sym os; os.p = fixed_syms + o; os.len = 1; if (allele_greater(cfix[o], os, c, me)) ++rank; }
            for (int t = head; t >= 0;) { const InsSlot sl = P.slots[t]; if (sl.count && ins_slot_greater(P, t, sl.count, c, me)) ++rank; t = sl.next; }
            if (rank == 0) { top_id = ch; top_c = c; }
            if (fixed_syms[ch] == refsym) { ref_key = ch; refc = c; reff = f; }
            else if (f >= P.min_freq_variants) { alt_fixed = 1; ++n_alt; }                        // 938-939
        }
        P.fixed_freq[gp * AMP_NCH + ch] = f; P.fixed_rank[gp * AMP_NCH + ch] = rank;
    }
    int s = head;
    for (int k = 0; k < ch && s >= 0; ++k) s = P.slots[s].next;
    for (int j = ch; s >= 0; j += G) {
        const int cs = P.slots[s].count;
        if (cs) {
            const Sym me = slot_sym(P, s);
            const double f = (double)cs / (double)total;
            int rank = 0;
AMP_UNROLL
            for (int o = 0; o < AMP_NCH; ++o)
                if (cfix[o]) { Sym os; os.p = fixed_syms + o; os.len = 1; if (allele_greater(cfix[o], os, cs, me)) ++rank; }
            for (int t = head; t >= 0;) { const InsSlot sl = P.slots[t]; if (t != s && sl.count && ins_slot_greater(P, t, sl.count, cs, me)) ++rank; t = sl.next; }
            const int kk = P.slot_entry[s];
            P.ins_freq[kk] = f; P.ins_rank[kk] = rank;
            if (rank == 0) { top_id = 6 + kk; top_c = cs; }
            unsigned char is_alt = 0;
            if (me.len == 1 && me.p[0] == refsym) { if (AMP_NCH + j > ref_key) { ref_key = AMP_NCH + j; refc = cs; reff = f; } }
            else if (f >= P.min_freq_variants) is_alt = 1;
            P.ins_alt[kk] = is_alt; n_alt += is_alt;
        }
        for (int k = 0; k < G && s >= 0; ++k) s = P.slots[s].next;
    }
    // position-level facts
    const unsigned lanes = (1u << G) - 1u;
    const unsigned top_m = (g_ballot(gmask, top_id >= 0) >> g0) & lanes;
    const unsigned alt_m = (g_ballot(gmask, alt_fixed != 0) >> g0) & lanes;
    const int top_l = top_m ? ffs32(top_m) - 1 : 0;
    top_id = g_shfl(gmask, top_id, g0 + top_l);
    top_c = g_shfl(gmask, top_c, g0 + top_l);
AMP_UNROLL
    for (int d = 1; d < G; d <<= 1) {
        n_alt += g_shfl_xor(gmask, n_alt, d);
        const int k2 = g_shfl_xor(gmask, ref_key, d);
        const int c2 = g_shfl_xor(gmask, refc, d);
        const double f2 = g_shfl_xor(gmask, reff, d);
        if (k2 > ref_key) { ref_key = k2; refc = c2; reff = f2; }
    }
    if (ch == 0) {
        P.depth[gp] = (int)total;
        P.top_id[gp] = top_m ? top_id : -1;
        P.top_count[gp] = top_m ? top_c : 0;
        unsigned char fl = 0;
        if (top_m) {
            const double bf = (double)top_c / (double)total;
            if (top_c >= P.min_depth_consensus && bf >= P.min_freq_consensus) fl |= 1;            // 928
        }
        if (total > 0 && total >= P.min_depth_variants && n_alt != 0) {                           // 940
            fl |= 2;
            if (refc >= P.min_depth_variants && reff >= P.min_freq_variants) fl |= 4;             // 948
        }
        P.pos_flags[gp] = fl; P.ref_count[gp] = refc; P.alt_mask[gp] = (unsigned char)(alt_m & 0x3Fu);
    }
}

// One position with insertion alleles, sixteen lanes: lanes 0..5 the fixed symbols A C G T N '-', lanes 6..15 the
// insertion alleles when there are at most ten (with more, call_long_list).  One float64 division per allele, the allele
// order (count, then python string order, descending: AmpliPy.py:771) from shuffles, the position-level facts from ballots.
// Every lane of the group takes part; fixed_syms has eight readable entries.
AMP_WD void call_group(const CallParams& P, const unsigned char* fixed_syms, long long gp, int sample, int p, int ch, int g0,
                            unsigned gmask) {
    constexpr int G = AMP_CALL_LANES, NINS = G - AMP_NCH;
    // (the fixed symbols' counts and the reference base are independent of the insertion list: loaded first, so that the latencies overlap)
    const int* cnt = P.counts + (size_t)sample * AMP_NCH * P.Lpad;
    const int c_fixed = ch < AMP_NCH ? cnt[(size_t)ch * P.Lpad + p] : 0;
    const unsigned char refsym = P.ref_seq[(size_t)sample * (size_t)P.ref_stride + p];
    // insertion alleles of the position: lane 6 + j takes the j-th entry of the list
    int slot = -1, s = P.heads[(size_t)sample * P.Lpad + p];
    for (int j = 0; j < NINS && s >= 0; ++j) {
        if (ch == AMP_NCH + j) slot = s;
        s = P.slots[s].next;
    }
    if (s >= 0) {                                             // longer list (uniform within the group)
        call_long_list(P, fixed_syms, gp, sample, p, ch, g0, gmask);
        return;
    }
    int c = c_fixed;
    Sym me; me.p = fixed_syms + (ch < AMP_NCH ? ch : 7); me.len = 1;
    if (ch >= AMP_NCH && slot >= 0) { c = P.slots[slot].count; me = slot_sym(P, slot); }
    int total = c;
AMP_UNROLL
    for (int d = 1; d < G; d <<= 1) total += g_shfl_xor(gmask, total, d);
    const double f = c ? (double)c / (double)total : 0.0;
    // index in the sorted allele list = number of alleles that are greater; only alleles that occur take part (one or two at most
    // positions), so the group walks the set bits of its occupancy mask instead of all sixteen lanes
    const unsigned lanes = (1u << G) - 1u;
    int rank = 0;
    for (unsigned occ = (g_ballot(gmask, c != 0) >> g0) & lanes; occ; occ &= occ - 1u) {
        const int o = ffs32(occ) - 1;
        const int co = g_shfl(gmask, c, g0 + o);
        Sym so;
        so.p = g_shfl(gmask, me.p, g0 + o);
        so.len = g_shfl(gmask, me.len, g0 + o);
        if (o != ch && c && allele_greater(co, so, c, me)) ++rank;
    }
    if (!c) rank = -1;
    const bool is_ref = c && me.len == 1 && me.p[0] == refsym;                     // 936-937
    const bool is_alt = c && !is_ref && f >= P.min_freq_variants;                  // 938-939
    const unsigned top_m = (g_ballot(gmask, rank == 0) >> g0) & lanes;
    const unsigned ref_m = (g_ballot(gmask, is_ref) >> g0) & lanes;
    const unsigned alt_m = (g_ballot(gmask, is_alt) >> g0) & lanes;
    const int best_l = top_m ? ffs32(top_m) - 1 : 0;
    const int best_c = g_shfl(gmask, c, g0 + best_l);
    const double best_f = g_shfl(gmask, f, g0 + best_l);
    const int kk = slot >= 0 ? P.slot_entry[slot] : -1;       // dense index of the insertion allele (amp_ins_export order)
    const int best_kk = g_shfl(gmask, kk, g0 + best_l);
    // the reference's loop visits the fixed symbols first, then the insertion alleles: the last match wins (936-937)
    const int ref_l = ref_m ? 31 - clz32(ref_m) : 0;
    const int refc0 = g_shfl(gmask, c, g0 + ref_l);
    const double reff0 = g_shfl(gmask, f, g0 + ref_l);
    if (ch < AMP_NCH) { P.fixed_freq[gp * AMP_NCH + ch] = f; P.fixed_rank[gp * AMP_NCH + ch] = rank; }
    else if (slot >= 0 && c) { P.ins_freq[kk] = f; P.ins_rank[kk] = rank; P.ins_alt[kk] = is_alt ? 1 : 0; }
    if (ch == 0) {
        const int refc = ref_m ? refc0 : 0;
        const double reff = ref_m ? reff0 : 0.0;
        P.depth[gp] = total;
        P.top_id[gp] = top_m ? (best_l < AMP_NCH ? best_l : 6 + best_kk) : -1;
        P.top_count[gp] = top_m ? best_c : 0;
        unsigned char fl = 0;
        if (top_m && best_c >= P.min_depth_consensus && best_f >= P.min_freq_consensus) fl |= 1;     // 928
        if (total > 0 && total >= P.min_depth_variants && alt_m != 0) {                             // 940
            fl |= 2;
            if (refc >= P.min_depth_variants && reff >= P.min_freq_variants) fl |= 4;               // 948
        }
        P.pos_flags[gp] = fl; P.ref_count[gp] = refc; P.alt_mask[gp] = (unsigned char)(alt_m & 0x3Fu);
    }
}

// thread t of the launch: lane t % 16 of the group of position t / 16 of the n_samples * L positions.  Groups never
// straddle warps; all sixteen lanes of a group call it.
AMP_HD void call_thread(const CallParams& P, const unsigned char* fixed_syms, long long t, int lane) {
    const long long gp = t / AMP_CALL_LANES;
    const int sample = (int)(gp / P.L), p = (int)(gp - (long long)sample * P.L);
    const int ch = lane & (AMP_CALL_LANES - 1), g0 = lane & AMP_CALL_LANES;
    call_group(P, fixed_syms, gp, sample, p, ch, g0, 0xFFFFu << g0);
}

}  // namespace amp
