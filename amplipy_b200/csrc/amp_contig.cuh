// amp_contig.cuh -- a batch grouped by contig (DESIGN.md 3.8): contig k of the FASTA is sample k of the context, and every
// contig's reads go through the fused kernel with that contig's own primer tables and length.  The fused kernels take one
// sample per launch, so a batch whose contigs are interleaved is first reordered into one contiguous range per contig.
// Written against the warp primitives of amp_warp.cuh, so that tests/emu runs this very source on the CPU.
//
//   contig_plan_cta      a tile of AMP_CT_TILE reads per CTA: the contig of every read (the BAM record's refID through a
//                        ref -> sample table, or an id the caller gives), a privatised per-contig histogram with the CIGAR-op
//                        and quality-byte totals, flushed with global atomics into one small table the host copies once
//   contig_scan_cta      one CTA: exclusive prefix sums of a u32 sequence (tile histograms in contig-major order, per-tile
//                        row totals)
//   contig_rank_cta      the stable counting sort: a read's place = its contig's base + the tile's earlier reads of that
//                        contig (per-warp histograms) + the rank among its warp's equal ids (__match_any_sync + popc)
//   contig_tilesum_cta   row totals (CIGAR ops, seq bytes, qual bytes) of each tile of the permuted order
//   contig_gather_cta    the permuted struct-of-arrays batch: scalars, re-scanned offsets, rows copied by a warp per read
//   contig_unpermute     the permuted launch's trim outputs back to input order
//   contig_skip          the trim outputs of reads without a contig (refID -1, flag 4), as the fused kernels write them (902)
#pragma once
#include "amp_bgzf.cuh"

namespace amp {

#define AMP_CT_THREADS 256        // threads of every CTA below
#define AMP_CT_TILE 2048          // reads per tile (eight per thread)
#define AMP_MAX_CONTIGS 1024      // what the plan's and the rank's shared histograms hold
#define AMP_CT_HDR 8              // header words of the plan table

#define AMP_CT_E_NOFLAG4 1        // a read without a contig (refID -1) that is not flagged unmapped (flag 4)
#define AMP_CT_E_UNKNOWN 2        // a read on a header sequence that is not in the FASTA
#define AMP_CT_E_BADID 4          // refID outside the header / sample id outside [-1, n_samples)

#if defined(__CUDA_ARCH__)
AMP_WD unsigned w_match(int v) { return __match_any_sync(0xFFFFFFFFu, v); }
AMP_WD void atomic_max64(unsigned long long* p, unsigned long long v) { atomicMax(p, v); }
#else
inline unsigned w_match(int v) {       // every lane of the warp takes part (the CTAs below keep whole warps in their loops)
    unsigned m = 0;
    for (int k = 0; k < 32; ++k) if (w_shfl(v, k) == v) m |= 1u << k;
    return m;
}
inline void atomic_max64(unsigned long long* p, unsigned long long v) { if (v > *p) *p = v; }
#endif
AMP_WD int low_lane(unsigned m) { return popc32((m & (0u - m)) - 1u); }

// Plan table, u64 words: [0] reads without a contig, [1] positions i > 0 whose contig differs from read i - 1's, [2] error
// bits, [3] CIGAR ops of the whole batch; then per contig k: reads at HDR + k, CIGAR ops at HDR + S + k, quality bytes at
// HDR + 2S + k, ~first read at HDR + 3S + k (a max of ~i is a min of i), cig_off[first] at HDR + 4S + k (written where a run of
// k starts: exact when the batch is grouped); then per header sequence r not in the FASTA, its reads at HDR + 5S + r.
AMP_HD size_t ct_table_words(int S, int n_refs) { return AMP_CT_HDR + 5 * (size_t)S + (size_t)(n_refs > 0 ? n_refs : 0); }

struct ContigPlanParams {
    long long n;
    const uint8_t* raw; const unsigned long long* rec_off;    // decoded batch: the inflated records ...
    const int* ref_to_sample; int n_refs;                     // ... and refID -> sample (-1: no contig, -2: not in the FASTA)
    const int* sample_in;                                     // or the sample of every read, given (-1: no contig)
    const uint16_t* flag; const uint32_t* cig_off; const uint32_t* qual_off;
    int S;
    int* sid;                          // [n] out: the contig of every read, -1 none, -2 error
    uint32_t* tile_hist;               // [n_tiles][S] out
    unsigned long long* table;         // zeroed by the caller
};

AMP_HD int contig_of(const ContigPlanParams& P, long long i, unsigned& err, int& unknown_ref) {
    int s;
    unknown_ref = -1;
    if (P.sample_in) {
        s = P.sample_in[i];
        if (s < -1 || s >= P.S) { err |= AMP_CT_E_BADID; return -2; }
    } else {
        const int rid = (int)ld_u32u(P.raw + P.rec_off[i] + 4);
        if (rid == -1) s = -1;
        else if (rid < -1 || rid >= P.n_refs) { err |= AMP_CT_E_BADID; return -2; }
        else {
            s = P.ref_to_sample[rid];
            if (s == -2) { err |= AMP_CT_E_UNKNOWN; unknown_ref = rid; return -2; }
            if (s < -1 || s >= P.S) { err |= AMP_CT_E_BADID; return -2; }
        }
    }
    if (s == -1 && !(P.flag[i] & 4)) err |= AMP_CT_E_NOFLAG4;
    return s;
}

struct ContigPlanSmem {
    int cnt[AMP_MAX_CONTIGS]; int fst[AMP_MAX_CONTIGS];
    unsigned long long cig[AMP_MAX_CONTIGS], qual[AMP_MAX_CONTIGS];
    unsigned long long all_cig; int nnc, nb; unsigned int err;
};

AMP_WD unsigned long long w_sum64(unsigned long long v) {      // over the whole warp (every lane takes part)
    const int lane = c_tid() & 31;
    for (int d = 16; d; d >>= 1) {
        const unsigned lo = (unsigned)w_shfl((int)(unsigned)v, lane ^ d), hi = (unsigned)w_shfl((int)(unsigned)(v >> 32), lane ^ d);
        v += ((unsigned long long)hi << 32) | lo;
    }
    return v;
}

// a thread takes AMP_CT_TILE / nthreads consecutive reads and adds each run of one contig to the tile's histogram at once; when
// the whole warp ends on one contig (a grouped batch), the warp adds its sums with one set of atomics
AMP_WD void contig_plan_cta(const ContigPlanParams& P, ContigPlanSmem& sm, int block) {
    const int tid = c_tid(), nt = c_nthreads(), S = P.S;
    unsigned long long* T = P.table;
    const long long r0 = (long long)block * AMP_CT_TILE, r1 = r0 + AMP_CT_TILE < P.n ? r0 + AMP_CT_TILE : P.n;
    for (int k = tid; k < S; k += nt) { sm.cnt[k] = 0; sm.fst[k] = 0x7FFFFFFF; sm.cig[k] = 0; sm.qual[k] = 0; }
    if (tid == 0) { sm.all_cig = 0; sm.nnc = 0; sm.nb = 0; sm.err = 0; }
    c_sync();
    const int per = AMP_CT_TILE / nt;
    const long long a = r0 + (long long)tid * per;
    unsigned err = 0;
    int nnc = 0, nb = 0, cur = -3, cnt = 0, prev = -3;
    long long first = 0;
    unsigned long long all_cig = 0, cig = 0, qual = 0;
    for (long long i = a; i < a + per && i < r1; ++i) {
        int uref, uprev;
        const int s = contig_of(P, i, err, uref);
        P.sid[i] = s;
        const uint32_t nc = P.cig_off[i + 1] - P.cig_off[i];
        all_cig += nc;
        if (uref >= 0) atomic_add64(&T[AMP_CT_HDR + 5 * (size_t)S + uref], 1ULL);
        if (i == a && i > 0) { unsigned e2 = 0; prev = contig_of(P, i - 1, e2, uprev); }
        const bool starts = i == 0 || prev != s;
        prev = s;
        if (starts && i > 0) ++nb;
        if (s >= 0) {
            if (s != cur) {
                if (cur >= 0) {
                    atomic_add(&sm.cnt[cur], cnt); atomic_min(&sm.fst[cur], (int)(first - r0));
                    atomic_add64(&sm.cig[cur], cig); atomic_add64(&sm.qual[cur], qual);
                }
                cur = s; cnt = 0; cig = 0; qual = 0; first = i;
            }
            ++cnt; cig += nc; qual += P.qual_off[i + 1] - P.qual_off[i];
            if (starts) T[AMP_CT_HDR + 4 * (size_t)S + s] = P.cig_off[i];
        } else if (s == -1) {
            ++nnc;
        }
    }
    const unsigned peers = w_match(cur);
    if (peers == 0xFFFFFFFFu && cur >= 0) {                          // the last runs of the whole warp are one contig's
        const int wcnt = w_add(cnt);
        const unsigned long long wcig = w_sum64(cig), wq = w_sum64(qual);
        long long f = first;
        for (int d = 16; d; d >>= 1) {
            const long long o = ((long long)(unsigned)w_shfl((int)(first >> 32), (tid & 31) ^ d) << 32) | (unsigned)w_shfl((int)first, (tid & 31) ^ d);
            f = o < f ? o : f;
            first = f;
        }
        if ((tid & 31) == 0) {
            atomic_add(&sm.cnt[cur], wcnt); atomic_min(&sm.fst[cur], (int)(f - r0));
            atomic_add64(&sm.cig[cur], wcig); atomic_add64(&sm.qual[cur], wq);
        }
    } else if (cur >= 0) {
        atomic_add(&sm.cnt[cur], cnt); atomic_min(&sm.fst[cur], (int)(first - r0));
        atomic_add64(&sm.cig[cur], cig); atomic_add64(&sm.qual[cur], qual);
    }
    const int wnnc = w_add(nnc), wnb = w_add(nb);
    const unsigned long long wall = w_sum64(all_cig);
    if ((tid & 31) == 0) {
        if (wnnc) atomic_add(&sm.nnc, wnnc);
        if (wnb) atomic_add(&sm.nb, wnb);
        if (wall) atomic_add64(&sm.all_cig, wall);
    }
    if (err) atomic_or(&sm.err, err);
    c_sync();
    for (int k = tid; k < S; k += nt) {
        P.tile_hist[(size_t)block * S + k] = (uint32_t)sm.cnt[k];
        if (sm.cnt[k]) {
            atomic_add64(&T[AMP_CT_HDR + k], (unsigned long long)sm.cnt[k]);
            atomic_add64(&T[AMP_CT_HDR + S + k], sm.cig[k]);
            atomic_add64(&T[AMP_CT_HDR + 2 * (size_t)S + k], sm.qual[k]);
            atomic_max64(&T[AMP_CT_HDR + 3 * (size_t)S + k], ~(unsigned long long)(r0 + sm.fst[k]));
        }
    }
    if (tid == 0) {
        if (sm.nnc) atomic_add64(&T[0], (unsigned long long)sm.nnc);
        if (sm.nb) atomic_add64(&T[1], (unsigned long long)sm.nb);
        if (sm.err) atomic_or((unsigned int*)&T[2], sm.err);         // the low word (little-endian)
        if (sm.all_cig) atomic_add64(&T[3], sm.all_cig);
    }
}

// ---- exclusive prefix sums of E u32 values (one CTA): value e is in[(e % inner) * s1 + (e / inner) * s2]; out has E + 1 entries
struct ContigScanParams {
    const uint32_t* in; long long E, inner, s1, s2;
    uint32_t* out;
};
AMP_HD uint32_t ct_scan_in(const ContigScanParams& P, long long e) { return P.in[(e % P.inner) * P.s1 + (e / P.inner) * P.s2]; }

// Hillis-Steele over one value per thread (part: nthreads u64); returns the exclusive prefix of v, *total = the sum
AMP_WD unsigned long long cta_excl_scan(unsigned long long v, unsigned long long* part, unsigned long long* total) {
    const int tid = c_tid(), nt = c_nthreads();
    part[tid] = v;
    c_sync();
    for (int d = 1; d < nt; d <<= 1) {
        const unsigned long long x = tid >= d ? part[tid - d] : 0ULL;
        c_sync();
        part[tid] += x;
        c_sync();
    }
    const unsigned long long incl = part[tid];
    *total = part[nt - 1];
    c_sync();
    return incl - v;
}

AMP_WD void contig_scan_cta(const ContigScanParams& P, unsigned long long* part) {
    const int tid = c_tid(), nt = c_nthreads();
    const long long per = (P.E + nt - 1) / nt, lo = tid * per, hi = lo + per < P.E ? lo + per : P.E;
    unsigned long long s = 0;
    for (long long e = lo; e < hi; ++e) s += ct_scan_in(P, e);
    unsigned long long total;
    unsigned long long run = cta_excl_scan(s, part, &total);
    for (long long e = lo; e < hi; ++e) { P.out[e] = (uint32_t)run; run += ct_scan_in(P, e); }
    if (tid == 0) P.out[P.E] = (uint32_t)total;
}

// ---- stable counting sort: perm[place] = read
struct ContigRankParams {
    long long n; int S; long long n_tiles;
    const int* sid;
    const uint32_t* hist_off;          // contig_scan_cta of tile_hist in contig-major order: [S][n_tiles]
    uint32_t* perm;
};
struct ContigRankSmem { int wc[AMP_CT_THREADS / 32][AMP_MAX_CONTIGS]; };

// warp w of the CTA takes the tile's reads [w * per, (w + 1) * per), 32 at a time; nthreads must be a multiple of 32
AMP_WD void contig_rank_cta(const ContigRankParams& P, ContigRankSmem& sm, int block) {
    const int tid = c_tid(), nt = c_nthreads(), lane = tid & 31, w = tid >> 5, nw = nt >> 5, S = P.S;
    const int per = AMP_CT_TILE / nw;
    const long long a = (long long)block * AMP_CT_TILE + (long long)w * per;
    for (int k = tid; k < nw * AMP_MAX_CONTIGS; k += nt) sm.wc[k / AMP_MAX_CONTIGS][k % AMP_MAX_CONTIGS] = 0;
    c_sync();
    for (int c = 0; c < per; c += 32) {                              // the warp's histogram
        const long long i = a + c + lane;
        const int s = i < P.n ? P.sid[i] : -3;
        const unsigned peers = w_match(s);
        if (s >= 0 && lane == low_lane(peers)) sm.wc[w][s] += popc32(peers);
        w_sync();
    }
    c_sync();
    for (int k = tid; k < S; k += nt) {                              // the place of each warp's first read of contig k
        unsigned run = P.hist_off[(size_t)k * P.n_tiles + block];
        for (int v = 0; v < nw; ++v) { const int x = sm.wc[v][k]; sm.wc[v][k] = (int)run; run += (unsigned)x; }
    }
    c_sync();
    for (int c = 0; c < per; c += 32) {
        const long long i = a + c + lane;
        const int s = i < P.n ? P.sid[i] : -3;
        const unsigned peers = w_match(s);
        const int base = s >= 0 ? sm.wc[w][s] : 0;
        if (s >= 0) P.perm[(unsigned)base + (unsigned)popc32(peers & ((1u << lane) - 1u))] = (uint32_t)i;
        w_sync();
        if (s >= 0 && lane == low_lane(peers)) sm.wc[w][s] = base + popc32(peers);
        w_sync();
    }
}

// ---- the permuted batch
struct ContigGatherParams {
    long long n, n_tiles;
    const uint32_t* perm;
    BatchPtrs src;                     // first = 0; seq may be null (no pileup)
    int32_t* pos; uint16_t* flag; int32_t* tlen; uint32_t* cig_off; uint32_t* cigar;
    uint32_t* seq_off; uint8_t* seq; uint32_t* qual_off; uint8_t* qual;
    uint32_t* tsum;                    // [n_tiles][3] CIGAR ops, seq bytes, qual bytes of each tile (contig_tilesum_cta)
    const uint32_t* tbase;             // [3][n_tiles + 1] their exclusive prefix sums
};
AMP_HD void ct_row_lens(const BatchPtrs& b, uint32_t i, uint32_t* len) {
    len[0] = b.cig_off[i + 1] - b.cig_off[i]; len[1] = b.seq_off[i + 1] - b.seq_off[i]; len[2] = b.qual_off[i + 1] - b.qual_off[i];
}

// thread t of the CTA owns the permuted reads [d0 + 8t, d0 + 8t + 8)
AMP_WD void contig_tilesum_cta(const ContigGatherParams& P, unsigned long long* part, int block) {
    const int tid = c_tid();
    const int per = AMP_CT_TILE / c_nthreads();
    const long long d0 = (long long)block * AMP_CT_TILE + (long long)tid * per;
    unsigned long long s[3] = {0, 0, 0};
    for (long long d = d0; d < d0 + per && d < P.n; ++d) {
        uint32_t len[3];
        ct_row_lens(P.src, P.perm[d], len);
        s[0] += len[0]; s[1] += len[1]; s[2] += len[2];
    }
    for (int ch = 0; ch < 3; ++ch) {
        unsigned long long total;
        cta_excl_scan(s[ch], part, &total);
        if (tid == 0) P.tsum[(size_t)block * 3 + ch] = (uint32_t)total;
    }
}

AMP_WD void contig_gather_cta(const ContigGatherParams& P, unsigned long long* part, int block) {
    const int tid = c_tid(), nt = c_nthreads(), lane = tid & 31, w = tid >> 5;
    const int per = AMP_CT_TILE / nt;
    const long long t0 = (long long)block * AMP_CT_TILE, d0 = t0 + (long long)tid * per;
    unsigned long long s[3] = {0, 0, 0};
    for (long long d = d0; d < d0 + per && d < P.n; ++d) {
        uint32_t len[3];
        ct_row_lens(P.src, P.perm[d], len);
        s[0] += len[0]; s[1] += len[1]; s[2] += len[2];
    }
    unsigned long long o[3];
    for (int ch = 0; ch < 3; ++ch) {
        unsigned long long total;
        o[ch] = P.tbase[(size_t)ch * (P.n_tiles + 1) + block] + cta_excl_scan(s[ch], part, &total);
    }
    for (long long d = d0; d < d0 + per && d < P.n; ++d) {
        const uint32_t i = P.perm[d];
        uint32_t len[3];
        ct_row_lens(P.src, i, len);
        P.cig_off[d] = (uint32_t)o[0]; P.seq_off[d] = (uint32_t)o[1]; P.qual_off[d] = (uint32_t)o[2];
        P.pos[d] = P.src.pos[i]; P.flag[d] = P.src.flag[i]; P.tlen[d] = P.src.tlen[i];
        o[0] += len[0]; o[1] += len[1]; o[2] += len[2];
        if (d == P.n - 1) { P.cig_off[P.n] = (uint32_t)o[0]; P.seq_off[P.n] = (uint32_t)o[1]; P.qual_off[P.n] = (uint32_t)o[2]; }
    }
    c_sync();
    // rows: a warp per read over the warp's 32 * per reads (stores of this CTA are visible after the barrier)
    const long long wa = t0 + (long long)w * 32 * per;
    for (long long d = wa; d < wa + 32 * per && d < P.n; ++d) {
        const uint32_t i = P.perm[d];
        uint32_t len[3];
        ct_row_lens(P.src, i, len);
        const uint32_t* cs = P.src.cigar + P.src.cig_off[i];
        uint32_t* cd = P.cigar + P.cig_off[d];
        for (uint32_t k = lane; k < len[0]; k += 32) cd[k] = cs[k];
        if (P.src.seq) {
            const uint8_t* ss = P.src.seq + P.src.seq_off[i];
            uint8_t* sd = P.seq + P.seq_off[d];
            for (uint32_t k = lane; k < len[1]; k += 32) sd[k] = ss[k];
        }
        const uint8_t* qs = P.src.qual + P.src.qual_off[i];
        uint8_t* qd = P.qual + P.qual_off[d];
        for (uint32_t k = lane; k < len[2]; k += 32) qd[k] = qs[k];
    }
}

// ---- trim outputs back to input order: row of permuted read d (at pcig_off[d] + 3d) -> row of read perm[d] (cig_off[i] + 3i)
struct ContigUnpermuteParams {
    long long n;
    const uint32_t* perm; const uint32_t* pcig_off; TrimOut po;
    const uint32_t* cig_off; TrimOut o;
};
AMP_WD void contig_unpermute_warp(const ContigUnpermuteParams& P, long long warp, long long n_warps) {
    const int lane = c_tid() & 31;
    for (long long d = warp; d < P.n; d += n_warps) {
        const uint32_t i = P.perm[d];
        const int nc = P.po.ncig[d];
        const uint32_t* src = P.po.cigar + (size_t)P.pcig_off[d] + 3 * (size_t)d;
        uint32_t* dst = P.o.cigar + (size_t)P.cig_off[i] + 3 * (size_t)i;
        for (int k = lane; k < nc; k += 32) dst[k] = src[k];
        if (lane == 0) { P.o.pos[i] = P.po.pos[d]; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = P.po.flags[d]; }
    }
}

// ---- reads without a contig: what the fused kernels write for a read that AmpliPy.py:902 skips
struct ContigSkipParams { long long n; const int* sid; BatchPtrs b; TrimOut o; };
AMP_HD void contig_skip_read(const ContigSkipParams& P, long long i) {
    if (P.sid[i] != -1) return;
    const uint32_t c0 = P.b.cig_off[i];
    const int nc = (int)(P.b.cig_off[i + 1] - c0);
    uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
    for (int k = 0; k < nc; ++k) orow[k] = P.b.cigar[c0 + k];
    P.o.pos[i] = P.b.pos[i]; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = (uint8_t)AMP_F_SKIPPED;
}

}  // namespace amp
