// amp_annot.cuh -- codon annotation of the iVar TSV (DESIGN.md 3.9): for every (sample, position) the (feature, codon) pairs
// the position belongs to, with the reference codon, its amino acid and the codon / amino acid of each substitution A C G T N.
// Written as __host__ __device__ code so that tests/emu runs this very source on the CPU.
//
//   annot_count   one thread per (sample, position): the number of its occurrences
//   (scan)        the counts -> CSR offsets [S*L + 1]
//   annot_fill    one thread per (sample, position): its occurrences at its offset, in (feature, spliced order), translated
//
// A sample's segments are kept sorted by genomic start with a running maximum of their ends: a position binary-searches the
// last segment that starts at or before it and walks back while the running maximum still reaches past it.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "amp_core.cuh"

namespace amp {

#define AMP_AN_THREADS 256
#define AMP_AN_NONE 0x7FFFFFFF

struct AnnotParams {
    int L, n_samples;
    const unsigned char* ref; long long ref_stride;    // the sample's reference starts at ref + sample * ref_stride
    const int* samp_seg;                                // [S + 1]: a sample's segments in the by-start arrays
    const int *sg_lo, *sg_max, *sg_key;                 // by start: start, running maximum of the ends, its spliced index
    const int *fs_lo, *fs_hi, *fs_cum, *fs_feat;        // spliced order (feature-major): [lo, hi), CDS bases before it, feature
    const int *ft_fs, *ft_len, *ft_local, *ft_info;     // per feature: [F + 1] spliced range, CDS length, index in its sample,
                                                        // phase | 4 for '-'
    unsigned int* off;                                  // [S*L + 1] CSR offsets (counts after annot_count)
    int *e_feat, *e_pos_aa;                             // per entry: feature index in its sample, 1-based codon index
    unsigned char* e_off;                               // offset of the position in the codon
    unsigned char* e_codon;                             // [E][18]: REF_CODON, then ALT_CODON for A C G T N
    unsigned char* e_aa;                                // [E][6]: REF_AA, then ALT_AA for A C G T N
};

// the standard genetic code (table 1), bases in the order T C A G
#define AMP_CODE1 "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"

AMP_HD int an_tcag(unsigned char b) { return b == 'T' ? 0 : b == 'C' ? 1 : b == 'A' ? 2 : b == 'G' ? 3 : -1; }
AMP_HD unsigned char an_upper(unsigned char b) { return b >= 'a' && b <= 'z' ? (unsigned char)(b - 32) : b; }
AMP_HD unsigned char an_comp(unsigned char b) {
    return b == 'A' ? 'T' : b == 'T' ? 'A' : b == 'C' ? 'G' : b == 'G' ? 'C' : 'N';
}
AMP_HD unsigned char an_translate(unsigned char b0, unsigned char b1, unsigned char b2) {
    const int x = an_tcag(b0), y = an_tcag(b1), z = an_tcag(b2);
    return (x | y | z) < 0 ? (unsigned char)'X' : (unsigned char)AMP_CODE1[16 * x + 4 * y + z];
}

// the spliced index of p in segment fs minus the phase (its place in the reading frame), or -1 when that base is skipped by
// the phase or lies in a trailing partial codon
AMP_HD int an_frame(const AnnotParams& P, int fs, int p) {
    const int f = P.fs_feat[fs], info = P.ft_info[f], phase = info & 3;
    const int within = (info & 4) ? P.fs_hi[fs] - 1 - p : p - P.fs_lo[fs];
    const int c = P.fs_cum[fs] + within - phase;
    return c >= 0 && c < (P.ft_len[f] - phase) / 3 * 3 ? c : -1;
}

// one past the last by-start segment of `sample` that starts at or before p
AMP_HD int an_upper_bound(const AnnotParams& P, int sample, int p) {
    int lo = P.samp_seg[sample], hi = P.samp_seg[sample + 1];
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (P.sg_lo[mid] <= p) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// the smallest spliced index > after of a segment that covers p with a complete codon there; AMP_AN_NONE if none.  A
// segment covers p when it starts at or before p and ends past it; fs_hi is read only where the running maximum says one may.
AMP_HD int an_next(const AnnotParams& P, int first, int top, int p, int after) {
    int best = AMP_AN_NONE;
    for (int i = top - 1; i >= first && P.sg_max[i] > p; --i) {
        const int fs = P.sg_key[i];
        if (fs > after && fs < best && P.fs_hi[fs] > p && an_frame(P, fs, p) >= 0) best = fs;
    }
    return best;
}

AMP_HD unsigned int annot_count(const AnnotParams& P, long long gp) {
    const int sample = (int)(gp / P.L), p = (int)(gp - (long long)sample * P.L);
    const int first = P.samp_seg[sample], top = an_upper_bound(P, sample, p);
    unsigned int n = 0;
    for (int i = top - 1; i >= first && P.sg_max[i] > p; --i) {
        const int fs = P.sg_key[i];
        n += P.fs_hi[fs] > p && an_frame(P, fs, p) >= 0;
    }
    return n;
}

// the reference base at spliced index t of feature f, upper-cased, in coding orientation
AMP_HD unsigned char an_base(const AnnotParams& P, const unsigned char* ref, int f, int t) {
    const bool minus = (P.ft_info[f] & 4) != 0;
    for (int fs = P.ft_fs[f]; fs < P.ft_fs[f + 1]; ++fs) {
        const int n = P.fs_hi[fs] - P.fs_lo[fs], d = t - P.fs_cum[fs];
        if (d < n) {
            const unsigned char b = an_upper(ref[minus ? P.fs_hi[fs] - 1 - d : P.fs_lo[fs] + d]);
            return minus ? an_comp(b) : b;
        }
    }
    return 'N';   // not reached: t < the feature's CDS length
}

// the occurrences of (sample, position) gp at entries [o, o + count), in spliced-index order (= feature order, then spliced order)
AMP_HD void annot_fill(const AnnotParams& P, long long gp, unsigned int o) {
    const int sample = (int)(gp / P.L), p = (int)(gp - (long long)sample * P.L);
    const int first = P.samp_seg[sample], top = an_upper_bound(P, sample, p);
    const unsigned char* ref = P.ref + (size_t)sample * (size_t)P.ref_stride;
    for (int fs = an_next(P, first, top, p, -1); fs != AMP_AN_NONE; fs = an_next(P, first, top, p, fs), ++o) {
        const int f = P.fs_feat[fs], c = an_frame(P, fs, p), k = c % 3, t0 = c - k + (P.ft_info[f] & 3);
        unsigned char cod[3];
        for (int j = 0; j < 3; ++j) cod[j] = an_base(P, ref, f, t0 + j);
        unsigned char* ec = P.e_codon + (size_t)o * 18;
        unsigned char* ea = P.e_aa + (size_t)o * 6;
        ec[0] = cod[0]; ec[1] = cod[1]; ec[2] = cod[2];
        ea[0] = an_translate(cod[0], cod[1], cod[2]);
        for (int a = 0; a < 5; ++a) {
            const unsigned char g = (unsigned char)"ACGTN"[a];
            const unsigned char b = (P.ft_info[f] & 4) ? an_comp(g) : g;
            unsigned char* x = ec + 3 + 3 * a;
            x[0] = k == 0 ? b : cod[0]; x[1] = k == 1 ? b : cod[1]; x[2] = k == 2 ? b : cod[2];
            ea[1 + a] = an_translate(x[0], x[1], x[2]);
        }
        P.e_feat[o] = P.ft_local[f]; P.e_pos_aa[o] = c / 3 + 1; P.e_off[o] = (unsigned char)k;
    }
}

// ---- host side: one sample's features as amp_set_features takes them, and the tables of AnnotParams for a context ---------
struct AnnotFeatures {
    std::vector<int> strand, phase, seg_off, lo, hi;    // segments of feature f: [seg_off[f], seg_off[f + 1]), 5' to 3'
};

// validates against the sample's length and orders each feature's segments 5' to 3' (ascending start on '+', descending on
// '-'); false on bad input
inline bool annot_features(int len, int n, const int32_t* strand, const int32_t* phase, const int32_t* seg_off, const int32_t* start,
                           const int32_t* end, AnnotFeatures& out) {
    if (n < 0 || (n > 0 && (!strand || !phase || !seg_off || !start || !end))) return false;
    out = AnnotFeatures();
    if (n == 0) return true;
    if (seg_off[0] != 0) return false;
    out.seg_off.push_back(0);
    for (int f = 0; f < n; ++f) {
        const int a = seg_off[f], b = seg_off[f + 1];
        if (b <= a || (strand[f] != 1 && strand[f] != -1) || phase[f] < 0 || phase[f] > 2) return false;
        std::vector<std::pair<int, int>> s;
        for (int k = a; k < b; ++k) {
            if (start[k] < 0 || end[k] <= start[k] || end[k] > len) return false;
            s.push_back({start[k], end[k]});
        }
        std::stable_sort(s.begin(), s.end(), [&](const std::pair<int, int>& x, const std::pair<int, int>& y) {
            return strand[f] > 0 ? x.first < y.first : x.first > y.first;
        });
        for (const auto& q : s) { out.lo.push_back(q.first); out.hi.push_back(q.second); }
        out.strand.push_back(strand[f]); out.phase.push_back(phase[f]); out.seg_off.push_back((int)out.lo.size());
    }
    return true;
}

struct AnnotTables {
    std::vector<int> samp_seg, sg_lo, sg_max, sg_key, fs_lo, fs_hi, fs_cum, fs_feat, ft_fs, ft_len, ft_local, ft_info;
};

// features of all samples -> the arrays of AnnotParams (features in sample order, then in the order given)
inline void annot_tables(const std::vector<AnnotFeatures>& samples, AnnotTables& T) {
    T = AnnotTables();
    T.samp_seg.push_back(0); T.ft_fs.push_back(0);
    for (const auto& s : samples) {
        const int fs0 = (int)T.fs_lo.size();
        for (size_t f = 0; f + 1 < s.seg_off.size(); ++f) {
            const int gf = (int)T.ft_len.size();
            int cum = 0;
            for (int k = s.seg_off[f]; k < s.seg_off[f + 1]; ++k) {
                T.fs_lo.push_back(s.lo[k]); T.fs_hi.push_back(s.hi[k]); T.fs_cum.push_back(cum); T.fs_feat.push_back(gf);
                cum += s.hi[k] - s.lo[k];
            }
            T.ft_fs.push_back((int)T.fs_lo.size()); T.ft_len.push_back(cum); T.ft_local.push_back((int)f);
            T.ft_info.push_back(s.phase[f] | (s.strand[f] < 0 ? 4 : 0));
        }
        const int fs1 = (int)T.fs_lo.size();
        std::vector<int> order;
        for (int k = fs0; k < fs1; ++k) order.push_back(k);
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return T.fs_lo[x] < T.fs_lo[y]; });
        int run = -1;
        for (int k : order) {
            run = T.fs_hi[k] > run ? T.fs_hi[k] : run;
            T.sg_lo.push_back(T.fs_lo[k]); T.sg_max.push_back(run); T.sg_key.push_back(k);
        }
        T.samp_seg.push_back((int)T.sg_lo.size());
    }
}

}  // namespace amp
