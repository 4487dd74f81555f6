// amp_emu_annot.cpp -- TEST INFRASTRUCTURE: the emulator of amp_emu_ivar.cpp plus the codon annotation of amp_annot.cuh (the
// per-position bodies of amp_annot_count_kernel / amp_annot_fill_kernel and the host-side tables), run on the CPU.
// Not part of the product.
#include "amp_emu_ivar.cpp"
#include "../../amplipy_b200/csrc/amp_annot.cuh"

namespace {
struct EmuAnnot {
    std::vector<unsigned int> off;
    std::vector<int> feat, pos_aa;
    std::vector<unsigned char> codon_off, codons, aas;
} g_annot;
}  // namespace

extern "C" {

// the features of S samples, sample s with nf[s] features: strand / phase per feature, seg_off[F + 1] over all features (a
// sample's slice is rebased, as amp_set_features receives it), segments start / end.  The tables as amp_annotate builds them,
// annot_count for every (sample, position), an exclusive scan, annot_fill.  Returns the number of entries, -1 on bad input
// (what amp_set_features returns AMP_ERR_ARG for).
long long emu_annot_build(int S, int L, const char* ref, long long ref_stride, const int* lens, const int* nf, const int* strand,
                          const int* phase, const int* seg_off, const int* start, const int* end) {
    std::vector<amp::AnnotFeatures> all((size_t)S);
    int f0 = 0;
    for (int s = 0; s < S; ++s) {
        std::vector<int> so((size_t)nf[s] + 1);
        for (int f = 0; f <= nf[s]; ++f) so[f] = seg_off[f0 + f] - seg_off[f0];
        const int k0 = seg_off[f0];
        if (!amp::annot_features(lens[s], nf[s], strand + f0, phase + f0, so.data(), start + k0, end + k0, all[s])) return -1;
        f0 += nf[s];
    }
    amp::AnnotTables T;
    amp::annot_tables(all, T);
    const long long SL = (long long)S * L;
    EmuAnnot& a = g_annot;
    a.off.assign((size_t)SL + 1, 0);
    amp::AnnotParams P{};
    P.L = L; P.n_samples = S; P.ref = (const unsigned char*)ref; P.ref_stride = ref_stride;
    P.samp_seg = T.samp_seg.data(); P.sg_lo = T.sg_lo.data(); P.sg_max = T.sg_max.data(); P.sg_key = T.sg_key.data();
    P.fs_lo = T.fs_lo.data(); P.fs_hi = T.fs_hi.data(); P.fs_cum = T.fs_cum.data(); P.fs_feat = T.fs_feat.data();
    P.ft_fs = T.ft_fs.data(); P.ft_len = T.ft_len.data(); P.ft_local = T.ft_local.data(); P.ft_info = T.ft_info.data();
    P.off = a.off.data();
    std::vector<unsigned int> cnt((size_t)SL);
    for (long long gp = 0; gp < SL; ++gp) cnt[gp] = amp::annot_count(P, gp);
    for (long long gp = 0; gp < SL; ++gp) a.off[gp + 1] = a.off[gp] + cnt[gp];
    const size_t E = a.off[SL];
    a.feat.assign(E + 1, -1); a.pos_aa.assign(E + 1, -1); a.codon_off.assign(E + 1, 255); a.codons.assign(18 * E + 1, 0);
    a.aas.assign(6 * E + 1, 0);
    P.e_feat = a.feat.data(); P.e_pos_aa = a.pos_aa.data(); P.e_off = a.codon_off.data(); P.e_codon = a.codons.data(); P.e_aa = a.aas.data();
    for (long long gp = 0; gp < SL; ++gp)
        if (cnt[gp]) amp::annot_fill(P, gp, a.off[gp]);
    return (long long)E;
}

// the last emu_annot_build's result, laid out as amp_annot_host copies it
void emu_annot_copy(uint32_t* off, int32_t* feat, int32_t* pos_aa, uint8_t* codon_off, uint8_t* codons, uint8_t* aas) {
    const EmuAnnot& a = g_annot;
    const size_t E = a.off.back();
    memcpy(off, a.off.data(), a.off.size() * 4);
    memcpy(feat, a.feat.data(), E * 4); memcpy(pos_aa, a.pos_aa.data(), E * 4); memcpy(codon_off, a.codon_off.data(), E);
    memcpy(codons, a.codons.data(), E * 18); memcpy(aas, a.aas.data(), E * 6);
}

}  // extern "C"
