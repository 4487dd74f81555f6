// amp_kernels.cuh -- CTA-level structure of the fused trim + pileup kernel and the calling kernel.
//
// The CTA body is written as barrier-separated phases over AMP_FOR_THREADS so that tests/emu can run
// the same source on the CPU (one loop over the CTA's threads per phase).  No warp collectives are
// used inside phases; cross-thread communication is shared-memory atomics + barriers only.
//
// Tile = up to `reads_per_tile` consecutive reads.  Per tile:
//   S  stage the tile's contiguous qual / seq byte ranges into shared memory (128-bit loads)
//   T  one thread per read: trim_read (AmpliPy.py:426-687), write trim outputs, plan the pileup
//      (update_base_counts, 690-753) into a shared list of aligned / deleted runs; insertion alleles
//      go to the global hash table
//   W  window decision: the CTA keeps a privatised counts tile cnt[6][WT] over reference window
//      [wbase, wbase+WT); when the tile's reads leave the window it is flushed with global atomics
//   C  one warp per run, lanes over consecutive bases: quality gate + base channel -> shared atomics
//      (channel-major tile with WT % 32 == 0 => 32 consecutive positions never bank-conflict)
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include "amp_core.cuh"

#if defined(__CUDA_ARCH__)
#define AMP_FOR_THREADS(tid, nthreads) for (int tid = threadIdx.x, once_ = 1; once_; once_ = 0)
#define AMP_SYNC() __syncthreads()
#ifdef AMP_PHASE_TIMING
#define AMP_TICK(k) do { if (threadIdx.x == 0) { long long t_ = clock64(); tacc[k] += t_ - tlast; tlast = t_; } } while (0)
#else
#define AMP_TICK(k) ((void)0)
#endif
#else
#define AMP_TICK(k) ((void)0)
#define AMP_FOR_THREADS(tid, nthreads) for (int tid = 0; tid < (nthreads); ++tid)
#define AMP_SYNC() ((void)0)
#endif

namespace amp {

struct BatchPtrs {
    long long first;         // global index of the first read to process (pointers are indexed with global indices)
    long long n;             // number of reads to process
    const int32_t* pos; const uint16_t* flag; const int32_t* tlen;
    const uint32_t* cig_off; const uint32_t* cigar;
    const uint32_t* seq_off; const uint8_t* seq;
    const uint32_t* qual_off; const uint8_t* qual;
};
struct TrimOut { int32_t* pos; uint16_t* ncig; uint8_t* flags; uint32_t* cigar; };

#define AMP_MODE_TRIM 1
#define AMP_MODE_PILEUP 2
#ifndef AMP_CMAX
#define AMP_CMAX 96      // CIGAR rows of up to 93 ops are rewritten in local memory (ONT-like reads: ~47 ops); longer ones in the global scratch
#endif

struct KParams {
    BatchPtrs b;
    TrimOut o;
    TrimParams tp;
    int mode;
    int* counts;             // [6][Lpad] of the sample being processed
    int Lpad;
    int gpos_base;           // sample * Lpad: position key used in the insertion table
    InsTable tab;
    unsigned int* err;
    uint32_t* scratch;       // 2 * (sumC + 3N) words, only touched by reads with n_cigar + 3 > AMP_CMAX
    long long scratch_half;  // sumC + 3N
    int reads_per_tile, ntiles, tiles_per_cta;
    int wt, maxseg, qbytes, sbytes;   // shared-memory carve-up
    int direct;                       // 1: launch the indel-rich kernel variant
    uint32_t* glist;                  // warp-autonomous kernel: per-CTA lists of the reads for its generic phase,
    long long gcap;                   //   gcap entries per CTA
    long long* phase_cycles;          // debug builds (-DAMP_PHASE_TIMING): per-CTA cycles in S, T, W, C
};

inline double amp_min_d(double a, double b) { return a < b ? a : b; }
inline double amp_max_d(double a, double b) { return a > b ? a : b; }
struct TileCfg { int wt, maxseg, qbytes, sbytes, reads_per_tile, direct; };

// shared-memory carve-up: three CTAs per SM at <= ~74 KB each (227 KB usable per SM).
// AMP_TILE="wt,maxseg,qbytes,sbytes,reads_per_tile" overrides it (tuning experiments only).
inline TileCfg pick_tile_cfg(long long n, long long sum_cig, long long sum_qual, int mode) {
    TileCfg t;
    const double avg_len = n ? (double)sum_qual / (double)n : 150.0;
    const double avg_ops = n ? (double)sum_cig / (double)n : 2.0;
    const bool indel_rich = avg_ops > 8.0;                                                         // ONT-like
    t.direct = indel_rich ? 1 : 0;
    // indel-rich: every read takes the per-thread generic path on rows read straight from the batch arrays and on work
    // rows in local memory, so what matters is how much of the SM's 256 KB stays L1: 28 KB per CTA (x 4 CTAs) leaves
    // 124 KB, the 44 KB of the former shape (1024, 512, 4096, 2048) left 60 KB and was 10 % slower
    if (indel_rich) { t.wt = 768; t.maxseg = 256; t.qbytes = 512; t.sbytes = 256; }
    else { t.wt = 512; t.maxseg = 512; t.qbytes = 33792; t.sbytes = 16896; }
    if (!(mode & AMP_MODE_PILEUP)) { t.wt = 32; t.maxseg = 16; t.sbytes = 16; t.qbytes = 40960; }
    double r = 256.0;
    if (!indel_rich) {
        r = amp_min_d(r, (double)t.qbytes * 0.97 / amp_max_d(avg_len, 1.0));
        if (mode & AMP_MODE_PILEUP) r = amp_min_d(r, (double)t.maxseg / (1.5 + 0.75 * avg_ops));
    }
    t.reads_per_tile = (int)amp_max_d(8.0, r);
#ifndef __CUDA_ARCH__
    if (const char* e = getenv("AMP_TILE")) {
        int a[5];
        if (sscanf(e, "%d,%d,%d,%d,%d", &a[0], &a[1], &a[2], &a[3], &a[4]) == 5) {
            t.wt = a[0]; t.maxseg = a[1]; t.qbytes = a[2]; t.sbytes = a[3]; t.reads_per_tile = a[4];
        }
    }
#endif
    return t;
}

#ifndef AMP_DEFER_MAX
#define AMP_DEFER_MAX 0      // >0: tiles with at most this many generic-path reads defer them to the end of the CTA
#endif                       // (measured slower on B200: in-tile they overlap with the counting warps; kept for experiments)
#define AMP_DLIST_CAP 384    // capacity of the per-CTA deferred list
#define AMP_DIRECT_MIN 32    // tiles with more generic-path reads than this count them thread-serially (DirectSink)
#define AMP_ROWS (AMP_NCH + 1)   // counts tile rows: 6 channels + one row that collects non-ACGTN bases (KeyError, 753)
AMP_HD size_t smem_bytes(int wt, int maxseg, int qbytes, int sbytes) {
    return (size_t)AMP_ROWS * wt * 4 + (size_t)maxseg * sizeof(Seg) + 128 + 512 + 4 * AMP_DLIST_CAP + (size_t)qbytes + (size_t)sbytes + 64;
}

struct Smem {
    int* cnt; Seg* segs; int* ctrl; uint8_t* qual; uint8_t* seq;
};
// ctrl words
// ctrl words: counters, nibble -> tile row LUT, C_CLIST: u16[256] reads of this tile queued for the generic path,
// C_DLIST: u32[AMP_DLIST_CAP] reads deferred to the end of the CTA
enum { C_NSEG = 0, C_TMIN = 1, C_TMAX = 2, C_NCPX = 3, C_LUT = 16, C_CLIST = 32, C_DLIST = 160 };

AMP_HD Smem carve(unsigned char* base, const KParams& P) {
    Smem s;
    s.cnt = (int*)base; base += (size_t)AMP_ROWS * P.wt * 4;
    s.segs = (Seg*)base; base += (size_t)P.maxseg * sizeof(Seg);
    s.ctrl = (int*)base; base += 128 + 512 + 4 * AMP_DLIST_CAP;
    s.qual = base; base += P.qbytes;
    s.seq = base;
    return s;
}

AMP_HD void count_add(const KParams& P, int* cnt, int wbase, int ch, int p) {
    const unsigned w = (unsigned)(p - wbase);
    if (wbase >= 0 && w < (unsigned)P.wt) atomic_add(&cnt[ch * P.wt + (int)w], 1);
    else atomic_add(&P.counts[(size_t)ch * P.Lpad + p], 1);
}

// privatised tile -> global count matrix; the extra row only raises the KeyError flag
AMP_HD void flush_tile(const KParams& P, int* cnt, int wbase, int tid, int nthreads, bool clear) {
    for (int ch = 0; ch < AMP_ROWS; ++ch) {
        for (int w = tid; w < P.wt; w += nthreads) {
            const int v = cnt[ch * P.wt + w];
            if (v) {
                if (ch < AMP_NCH) atomic_add(&P.counts[(size_t)ch * P.Lpad + wbase + w], v);
                else atomic_or(P.err, AMP_E_BASE);
                if (clear) cnt[ch * P.wt + w] = 0;
            }
        }
    }
}

// Per-read sink used in phase T.
struct TileSink {
    const KParams* P; Smem sm;
    uint32_t qabs0, nibabs0;           // first quality byte / first nibble of this read: staging-buffer relative when
    bool staged;                       // `staged` (both rows fit the staging buffers), else absolute in the batch arrays
    const uint8_t* seq_read;           // this read's packed sequence (shared or global)
    const uint8_t* qual_read;
    unsigned int errs;
    AMP_HD void push(int rpos, int len_kind, int q) {
        int idx = atomic_add(&sm.ctrl[C_NSEG], 1);
        if (idx < P->maxseg) {
            Seg s; s.rpos = rpos; s.len = len_kind | (staged ? 0x40000000 : 0); s.qabs = qabs0 + (uint32_t)q; s.nibabs = nibabs0 + (uint32_t)q;
            sm.segs[idx] = s;
        } else {
            // list full: count this run serially, straight into the global matrix (exact, slow, rare)
            const int n = len_kind & 0x3FFFFFFF;
            if (len_kind < 0) { for (int j = 0; j < n; ++j) atomic_add(&P->counts[(size_t)5 * P->Lpad + rpos + j], 1); }
            else for (int j = 0; j < n; ++j) {
                if (qual_read[q + j] < P->tp.min_quality) continue;
                int ch = nib_channel(nib_at(seq_read, (uint32_t)(q + j)));
                if (ch < 0) { errs |= AMP_E_BASE; continue; }
                atomic_add(&P->counts[(size_t)ch * P->Lpad + rpos + j], 1);
            }
        }
    }
    AMP_HD void match(int rpos, int q, int n) { push(rpos, n, q); }
    AMP_HD void del(int rpos, int n, int /*qa*/) { push(rpos, (int)(0x80000000u | (unsigned)n), 0); }
    struct Text {
        const uint8_t* seq; int b;
        AMP_HD char operator()(int i) const { return nib_char(nib_at(seq, (uint32_t)(b + i))); }
        AMP_HD uint32_t word(int i, int len) const {
            // three independent byte loads cover the four nibbles wherever they start; none beyond the key's last byte
            const uint32_t idx = (uint32_t)(b + i);
            const uint8_t* a = seq + (idx >> 1);
            const uint32_t m = len - i < 4 ? (uint32_t)(len - i) : 4u;
            const uint32_t nb = ((idx + m - 1u) >> 1) - (idx >> 1);        // bytes after a[0] that hold key nibbles (0..2)
            const uint32_t x = ((uint32_t)a[0] << 16) | ((nb >= 1u ? (uint32_t)a[1] : 0u) << 8) | (nb >= 2u ? (uint32_t)a[2] : 0u);
            const uint32_t y = x >> ((idx & 1u) ? 4 : 8);              // nibbles idx .. idx+3 in bits 15..0, first one on top
            uint32_t w = nib_pair_chars(y >> 8) | (nib_pair_chars(y) << 16);
            if (len - i < 4) w &= (1u << (8 * (len - i))) - 1u;
            return w;
        }
    };
    AMP_HD void ins(int pos, int b, int n, int /*q0*/ = 0) {
        if (n == 1) {   // one-character key == that base's own dict entry (AmpliPy.py:745-746)
            int ch = nib_channel(nib_at(seq_read, (uint32_t)b));
            if (ch >= 0) { atomic_add(&P->counts[(size_t)ch * P->Lpad + pos], 1); return; }
        }
        Text t; t.seq = seq_read; t.b = b;
        ins_table_add(P->tab, P->gpos_base + pos, n, t, 1);
    }
};

// Pull the next tile's inputs towards L2 while the current tile is being processed (one 128-byte line per
// thread and array); purely a hint, so the emulation build leaves it out.
AMP_HD void prefetch_tile(const KParams& P, long long t0, int tid, int nthreads) {
#ifdef __CUDA_ARCH__
    long long t1 = t0 + P.reads_per_tile; if (t1 > P.b.first + P.b.n) t1 = P.b.first + P.b.n;
    if (t1 <= t0) return;
    auto pf = [&](const void* base, size_t lo, size_t hi) {
        const char* p0 = (const char*)base + (lo & ~(size_t)127);
        const char* p1 = (const char*)base + hi;
        for (const char* p = p0 + (size_t)tid * 128; p < p1; p += (size_t)nthreads * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    };
    const size_t q0 = P.b.qual_off[t0], q1 = P.b.qual_off[t1];
    pf(P.b.qual, q0, q1);
    if (P.mode & AMP_MODE_PILEUP) pf(P.b.seq, P.b.seq_off[t0], P.b.seq_off[t1]);
    pf(P.b.cigar, (size_t)P.b.cig_off[t0] * 4, (size_t)P.b.cig_off[t1] * 4);
    pf(P.b.pos, (size_t)t0 * 4, (size_t)t1 * 4);
    pf(P.b.tlen, (size_t)t0 * 4, (size_t)t1 * 4);
    pf(P.b.flag, (size_t)t0 * 2, (size_t)t1 * 2);
#else
    (void)P; (void)t0; (void)tid; (void)nthreads;
#endif
}

// Sink for tiles that are mostly generic-path reads (indel-rich data, e.g. ONT): the planning thread counts its
// own runs base by base into the CTA's tile.  A run list would hold tens of short runs per read, and one warp per
// ~10-base run wastes most lanes; here all lanes of the warp stay busy, each on its own read.
struct DirectSink {
    const KParams* P; Smem sm; int wbase;
    const uint8_t* seq_read; const uint8_t* qual_read;
    unsigned int errs;
    AMP_HD void match(int rpos, int q, int n) {
        const int* lut = sm.ctrl + C_LUT;
        const int minq = P->tp.min_quality;
        const int w0 = rpos - wbase;
        if (wbase >= 0 && w0 >= 0 && w0 + n <= P->wt) {
            int* c = sm.cnt + w0;
            for (int j = 0; j < n; ++j) {
                if (qual_read[q + j] < minq) continue;                                   // AmpliPy.py:718
                atomic_add(c + j + lut[nib_at(seq_read, (uint32_t)(q + j))], 1);         // 752-753 (row 6 = KeyError flag)
            }
        } else {
            for (int j = 0; j < n; ++j) {
                if (qual_read[q + j] < minq) continue;
                const int ch = nib_channel(nib_at(seq_read, (uint32_t)(q + j)));
                if (ch < 0) { errs |= AMP_E_BASE; continue; }
                count_add(*P, sm.cnt, wbase, ch, rpos + j);
            }
        }
    }
    AMP_HD void del(int rpos, int n, int /*qa*/ = -1) { for (int j = 0; j < n; ++j) count_add(*P, sm.cnt, wbase, 5, rpos + j); }   // 714-715
    AMP_HD void ins(int pos, int b, int n, int /*q0*/ = 0) {
        if (n == 1) {
            int ch = nib_channel(nib_at(seq_read, (uint32_t)b));
            if (ch >= 0) { atomic_add(&P->counts[(size_t)ch * P->Lpad + pos], 1); return; }
        }
        TileSink::Text t; t.seq = seq_read; t.b = b;
        ins_table_add(P->tab, P->gpos_base + pos, n, t, 1);
    }
};

// DirectSink in two steps.  Lanes of a warp reach the runs and insertions of their reads at different points of
// plan_read's CIGAR walk, so counting inside the walk runs a lane or two at a time (ncu on ONT-like batches: 1.9
// active lanes in the count loop, 1.1 in the insertion-table code).  Here the walk only records what it finds in
// per-thread lists; replay() then counts every base of the read in one flat loop and adds the insertion alleles in
// another, with the lanes of the warp together again.  Whatever does not fit a list takes DirectSink's immediate path.
#ifndef AMP_REC_RUNS
#define AMP_REC_RUNS 64
#endif
#ifndef AMP_REC_INS
#define AMP_REC_INS 24
#endif
struct RecordSink {
    DirectSink d;
    int rp[AMP_REC_RUNS]; uint32_t ql[AMP_REC_RUNS];   // run: first reference position; (query index << 16) | deletion << 15 | length
    int ip[AMP_REC_INS]; uint32_t ib[AMP_REC_INS];     // insertion allele: position; (first base << 16) | length
    int nrun, nins, steps;
    AMP_HD void match(int rpos, int q, int n) {
        if (nrun < AMP_REC_RUNS && q < 65536 && n < 32768) { rp[nrun] = rpos; ql[nrun] = ((uint32_t)q << 16) | (uint32_t)n; ++nrun; steps += n; }
        else d.match(rpos, q, n);
    }
    AMP_HD void del(int rpos, int n, int /*qa*/) {
        if (nrun < AMP_REC_RUNS && n < 32768) { rp[nrun] = rpos; ql[nrun] = 0x8000u | (uint32_t)n; ++nrun; steps += n; }
        else d.del(rpos, n);
    }
    AMP_HD void ins(int pos, int b, int n, int /*q0*/ = 0) {
        if (nins < AMP_REC_INS && b < 65536 && n < 65536) { ip[nins] = pos; ib[nins] = ((uint32_t)b << 16) | (uint32_t)n; ++nins; }
        else d.ins(pos, b, n);
    }
    // cnt / lut: the CTA's tile and nibble -> row table, passed by the caller so that they stay shared-memory pointers
    // (this struct lives in local memory: pointers read back from it would be generic, and so would the atomics)
    AMP_HD void replay(const KParams& P, int* cnt, const int* lut, int wbase, const uint8_t* seq_read, const uint8_t* qual_read) {
        const int minq = P.tp.min_quality, wt = P.wt;
        int k = -1, j = 0, n = 0, rpos = 0, q = 0;
        bool is_del = false, in_win = false;
        for (int t = 0; t < steps; ++t, ++j) {
            if (j == n) {                                                                 // next run (lengths are > 0)
                ++k;
                const uint32_t w = ql[k];
                rpos = rp[k]; n = (int)(w & 0x7FFFu); q = (int)(w >> 16); is_del = (w & 0x8000u) != 0; j = 0;
                in_win = wbase >= 0 && rpos >= wbase && rpos + n <= wbase + wt;
            }
            const int p = rpos + j;
            if (is_del) {                                                                 // 714-715
                if (in_win) atomic_add(cnt + 5 * wt + (p - wbase), 1); else atomic_add(&P.counts[(size_t)5 * P.Lpad + p], 1);
                continue;
            }
            if (qual_read[q + j] < minq) continue;                                        // 718
            const uint32_t nib = nib_at(seq_read, (uint32_t)(q + j));
            if (in_win) { atomic_add(cnt + (p - wbase) + lut[nib], 1); continue; }        // 752-753 (row 6 = KeyError flag)
            const int ch = nib_channel(nib);
            if (ch < 0) { d.errs |= AMP_E_BASE; continue; }
            atomic_add(&P.counts[(size_t)ch * P.Lpad + p], 1);
        }
        for (int e = 0; e < nins; ++e) d.ins(ip[e], (int)(ib[e] >> 16), (int)(ib[e] & 0xFFFFu));
    }
};

// Everything a thread needs to know about the tile it is working on.
struct TileCtx {
    long long t0; int nreads;
    uint32_t q_lo, q_hi, s_lo, s_hi;   // staged byte ranges [lo, hi) of qual / seq
    uint32_t q_glo, q_ghi;             // byte range of the launch's qualities in the batch array
    bool do_trim, do_pile;
};

// Generic per-read path: trim_read loop for loop + plan_read.  Used for every read that is not [S]M[S]
// (indels, hard clips, ...) and for the corner cases the closed form declines.
template <bool DIRECT>
AMP_HD void read_generic(const KParams& P, const Smem& sm, const TileCtx& T, int rr, bool direct, int wbase) {
    const long long i = T.t0 + rr;
#ifdef __CUDA_ARCH__
    const unsigned lanes = __activemask();     // the lanes that entered together
#define AMP_RECONVERGE(m) __syncwarp(m)
#else
    const unsigned lanes = 0;
#define AMP_RECONVERGE(m) ((void)0)
#endif
    const uint32_t c0 = P.b.cig_off[i], c1 = P.b.cig_off[i + 1];
    const uint32_t qo0 = P.b.qual_off[i], qo1 = P.b.qual_off[i + 1];
    const uint32_t so0 = P.b.seq_off[i], so1 = P.b.seq_off[i + 1];
    int nc = (int)(c1 - c0);
    const int l_seq = (int)(qo1 - qo0);
    const int flag = P.b.flag[i];
    int pos = P.b.pos[i];
    const bool q_st = qo1 <= T.q_hi, s_st = T.do_pile && so1 <= T.s_hi;
    const uint8_t* qual = q_st ? sm.qual + (qo0 - T.q_lo) : P.b.qual + qo0;
    const uint8_t* seq = s_st ? sm.seq + (so0 - T.s_lo) : P.b.seq + so0;
    const uint32_t* cig = P.b.cigar + c0;
    uint32_t la[AMP_CMAX], lb[AMP_CMAX];
    int f = 0;
    if (T.do_trim) {
        uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
        uint32_t *A, *B;
        if (nc + 3 <= AMP_CMAX) { A = la; B = lb; }
        else { A = P.scratch + (size_t)c0 + 3 * (size_t)i; B = A + P.scratch_half; }
        for (int k = 0; k < nc; ++k) A[k] = cig[k];
        uint32_t* res;
        // word-wise window search: staged rows have slack around them; rows read from the batch array have their
        // neighbours' bytes, except within 8 bytes of the start / 16 of the end of the launch's range
        const bool q_pad = q_st || (qo0 >= T.q_glo + 8u && qo1 + 16u <= T.q_ghi);
        f = trim_read(A, B, nc, pos, flag, P.b.tlen[i], l_seq, qual, q_pad, P.tp, &res, lanes);
        if (f & AMP_F_ERROR) { nc = 0; f = AMP_F_ERROR; atomic_or(P.err, AMP_E_COORD); }
        for (int k = 0; k < nc; ++k) orow[k] = res[k];
        cig = res;
        P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = (uint8_t)f;
    }
    AMP_RECONVERGE(lanes);
    if (DIRECT && T.do_pile && direct) {                  // uniform over the tile
        RecordSink sink;
        sink.d.P = &P; sink.d.sm = sm; sink.d.wbase = wbase; sink.d.seq_read = seq; sink.d.qual_read = qual; sink.d.errs = 0;
        sink.nrun = sink.nins = sink.steps = 0;
        int e = 0;
        if (!(f & AMP_F_ERROR)) e = plan_read(cig, nc, pos, l_seq, qual, P.tp.min_quality, P.tp.L, sink);
        AMP_RECONVERGE(lanes);
        sink.replay(P, sm.cnt, sm.ctrl + C_LUT, wbase, seq, qual);
        e |= (int)sink.d.errs;
        if (e) atomic_or(P.err, (unsigned)e);
    } else if (T.do_pile && !(f & AMP_F_ERROR)) {
        TileSink sink; sink.P = &P; sink.sm = sm;
        sink.staged = q_st && s_st;
        sink.qabs0 = sink.staged ? qo0 - T.q_lo : qo0;
        sink.nibabs0 = sink.staged ? (so0 - T.s_lo) * 2u : so0 * 2u;
        sink.seq_read = seq; sink.qual_read = qual; sink.errs = 0;
        int e = plan_read(cig, nc, pos, l_seq, qual, P.tp.min_quality, P.tp.L, sink);
        e |= (int)sink.errs;
        if (e) atomic_or(P.err, (unsigned)e);
        if (!(e & (AMP_E_COORD | AMP_E_CIGAR))) { atomic_min(&sm.ctrl[C_TMIN], pos); atomic_max(&sm.ctrl[C_TMAX], pos + ref_len_of(cig, nc)); }
    }
}

// Count phase over runs [lo, hi) of the tile's list.  A warp works on 32/AMP_SUBWARP runs at once: each group of
// AMP_SUBWARP lanes takes one run and steps over it AMP_SUBWARP consecutive bases at a time.  Runs after trimming
// average ~75 bases, so narrower groups waste fewer lanes on the last step and share the per-run set-up across
// several runs; within a group consecutive lanes still hit consecutive banks of one tile row.
// Warps [0, skip_warps) do not take part (they are busy with the generic path of queued reads).
#ifndef AMP_SUBWARP
#define AMP_SUBWARP 8
#endif
AMP_HD void count_runs(const KParams& P, const Smem& sm, int lo, int hi, int wbase, int tid, int nthreads, int skip_warps) {
    constexpr int SW = AMP_SUBWARP, GROUPS = 32 / SW;
    const int lane = tid & 31, l = lane % SW, sub = lane / SW;
    int warp = tid >> 5, nwarps = nthreads >> 5 ? nthreads >> 5 : 1;
    if (skip_warps >= nwarps) skip_warps = 0;
    if (warp < skip_warps) return;
    warp -= skip_warps; nwarps -= skip_warps;
    const int* lut = sm.ctrl + C_LUT;
    const int minq = P.tp.min_quality;
    unsigned errs = 0;
    for (int s = lo + (warp % nwarps) * GROUPS + sub; s < hi; s += nwarps * GROUPS) {
        const Seg sg = sm.segs[s];
        const int n = sg.len & 0x3FFFFFFF;
        const int w0 = sg.rpos - wbase;
        const bool in_win = wbase >= 0 && w0 >= 0 && w0 + n <= P.wt;                // uniform per run
        if (sg.len < 0) {
            if (in_win) { for (int j = l; j < n; j += SW) atomic_add(&sm.cnt[5 * P.wt + w0 + j], 1); }
            else for (int j = l; j < n; j += SW) count_add(P, sm.cnt, wbase, 5, sg.rpos + j);
            continue;
        }
        const bool staged = (sg.len & 0x40000000) != 0;
        if (in_win && staged) {
            // fast path: everything in shared memory, no per-base branches.  Tail lanes (j >= n) read at most
            // SW-1 bytes past the run, which stays inside the padded staging buffers; the predicate discards them.
            const uint8_t* q = sm.qual + sg.qabs + l;
            const uint32_t nb0 = sg.nibabs + (uint32_t)l;
            const uint32_t shift = (~nb0 & 1u) << 2;
            const uint8_t* sb = sm.seq + (nb0 >> 1);
            int* c = sm.cnt + w0 + l;
            const int left = n - l;                                                // this lane has bases l, l+SW, ... < n
            const int iters = (n + SW - 1) / SW;
#if defined(__CUDA_ARCH__)
#pragma unroll 4
#endif
            for (int u = 0; u < iters; ++u) {
                const int qv = q[SW * u];
                const uint32_t nib = ((uint32_t)sb[(SW / 2) * u] >> shift) & 15u;
                const int row = lut[nib];
                if (left > SW * u && qv >= minq) atomic_add(c + SW * u + row, 1);   // AmpliPy.py:718, 752-753
            }
        } else {
            const uint8_t* qp = staged ? sm.qual + sg.qabs : P.b.qual + sg.qabs;
            const uint8_t* sp = staged ? sm.seq : P.b.seq;
            for (int j = l; j < n; j += SW) {
                if (qp[j] < minq) continue;
                const uint32_t nb = sg.nibabs + (uint32_t)j;
                const int ch = nib_channel((sp[nb >> 1] >> ((~nb & 1u) << 2)) & 15u);
                if (ch < 0) { errs |= AMP_E_BASE; continue; }
                count_add(P, sm.cnt, wbase, ch, sg.rpos + j);
            }
        }
    }
    if (errs) atomic_or(P.err, errs);
}

// The fused CTA body.  `block` / `nthreads` are blockIdx.x / blockDim.x on the device.  DIRECT = variant for
// indel-rich batches (generic-path reads count their own runs, DirectSink); the two variants are separate kernels so
// that the common short-read kernel does not carry the extra code.
template <bool DIRECT>
AMP_HD void cta_trim_pileup(const KParams& P, unsigned char* smem_base, int block, int nthreads) {
    const Smem sm = carve(smem_base, P);
    const bool do_trim = P.mode & AMP_MODE_TRIM, do_pile = P.mode & AMP_MODE_PILEUP;
    const int ncnt = AMP_ROWS * P.wt;
    int wbase = -1;                                    // uniform across the CTA
#if defined(__CUDA_ARCH__) && defined(AMP_PHASE_TIMING)
    long long tacc[4] = {0, 0, 0, 0}, tlast = clock64();
#endif
    if (do_pile) {
        AMP_FOR_THREADS(tid, nthreads) {
            for (int i = tid; i < ncnt; i += nthreads) sm.cnt[i] = 0;
            if (tid < 16) { const int ch = nib_channel((uint32_t)tid); sm.ctrl[C_LUT + tid] = (ch < 0 ? AMP_NCH : ch) * P.wt; }
        }
    }
    uint16_t* clist = (uint16_t*)(sm.ctrl + C_CLIST);
    uint32_t* dlist = (uint32_t*)(sm.ctrl + C_DLIST);   // reads deferred to the end of the CTA (absolute index - P.b.first)
    int ndef = 0;                                        // uniform
    (void)dlist; (void)ndef;
    const int tile_lo = block * P.tiles_per_cta;
    int tile_hi = tile_lo + P.tiles_per_cta; if (tile_hi > P.ntiles) tile_hi = P.ntiles;
    for (int tile = tile_lo; tile < tile_hi; ++tile) {
        TileCtx T;
        T.t0 = P.b.first + (long long)tile * P.reads_per_tile;
        long long t1 = T.t0 + P.reads_per_tile; if (t1 > P.b.first + P.b.n) t1 = P.b.first + P.b.n;
        T.nreads = (int)(t1 - T.t0); T.do_trim = do_trim; T.do_pile = do_pile;
        T.q_glo = P.b.qual_off[P.b.first]; T.q_ghi = P.b.qual_off[P.b.first + P.b.n];
        // ---- S: stage qual / seq of the tile ------------------------------------------------------
        const uint32_t q_end = P.b.qual_off[t1], s_end = P.b.seq_off[t1];
        T.q_lo = P.b.qual_off[T.t0] & ~15u; T.s_lo = P.b.seq_off[T.t0] & ~15u;
        T.q_hi = (q_end - T.q_lo <= (uint32_t)P.qbytes) ? q_end : T.q_lo + (uint32_t)P.qbytes;   // staged [lo, hi)
        T.s_hi = (s_end - T.s_lo <= (uint32_t)P.sbytes) ? s_end : T.s_lo + (uint32_t)P.sbytes;
        AMP_FOR_THREADS(tid, nthreads) {
            if (tid == 0) { sm.ctrl[C_NSEG] = 0; sm.ctrl[C_TMIN] = 0x7FFFFFFF; sm.ctrl[C_TMAX] = -1; sm.ctrl[C_NCPX] = 0; }
            {
                const uint32_t nvec = (T.q_hi - T.q_lo) >> 4;
                const uint4* g = (const uint4*)(P.b.qual + T.q_lo); uint4* s = (uint4*)sm.qual;
                for (uint32_t v = tid; v < nvec; v += nthreads) s[v] = g[v];
                for (uint32_t k = (nvec << 4) + tid; k < T.q_hi - T.q_lo; k += nthreads) sm.qual[k] = P.b.qual[T.q_lo + k];
            }
            if (do_pile) {
                const uint32_t nvec = (T.s_hi - T.s_lo) >> 4;
                const uint4* g = (const uint4*)(P.b.seq + T.s_lo); uint4* s = (uint4*)sm.seq;
                for (uint32_t v = tid; v < nvec; v += nthreads) s[v] = g[v];
                for (uint32_t k = (nvec << 4) + tid; k < T.s_hi - T.s_lo; k += nthreads) sm.seq[k] = P.b.seq[T.s_lo + k];
            }
        }
        AMP_SYNC(); AMP_TICK(0);
        // ---- T0: one thread per read.  [S]M[S] reads are finished here in registers (closed-form trim, one
        // aligned run); everything else is queued for the generic path.
        AMP_FOR_THREADS(tid, nthreads) {
            if (tile + 1 < tile_hi) prefetch_tile(P, t1, tid, nthreads);   // overlaps this tile's compute phases
            for (int rr = tid; rr < T.nreads; rr += nthreads) {
                const long long i = T.t0 + rr;
                const uint32_t c0 = P.b.cig_off[i], c1 = P.b.cig_off[i + 1];
                const uint32_t qo0 = P.b.qual_off[i], qo1 = P.b.qual_off[i + 1];
                const int nc = (int)(c1 - c0), l_seq = (int)(qo1 - qo0);
                const int flag = P.b.flag[i];
                int pos = P.b.pos[i];
                const uint32_t* cig = P.b.cigar + c0;
                if ((flag & 4) || nc == 0) {                                            // AmpliPy.py:902
                    if (do_trim) {
                        uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
                        for (int k = 0; k < nc; ++k) orow[k] = cig[k];
                        P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = (uint8_t)AMP_F_SKIPPED;
                    }
                    continue;
                }
                SimpleRead r;
                const bool q_st = qo1 <= T.q_hi;
                bool done = q_st && rr < 65536 && classify_simple(cig, nc, l_seq, r);
                int f = 0;
                if (done && do_trim) done = trim_simple(r, pos, flag, P.b.tlen[i], l_seq, sm.qual + (qo0 - T.q_lo), true, P.tp, &f);
                if (done && !do_trim && (pos < 0 || pos + r.m > P.tp.L)) done = false;
                if (done) {
                    if (do_trim) {
                        uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
                        const int no = emit_simple(r, orow);
                        P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)no; P.o.flags[i] = (uint8_t)f;
                    }
                    if (do_pile && r.m > 0) {
                        const uint32_t so0 = P.b.seq_off[i], so1 = P.b.seq_off[i + 1];
                        const bool staged = so1 <= T.s_hi;                            // q_st holds
                        const int idx = atomic_add(&sm.ctrl[C_NSEG], 1);
                        if (idx < P.maxseg) {
                            Seg sgm; sgm.rpos = pos; sgm.len = r.m | (staged ? 0x40000000 : 0);
                            sgm.qabs = (staged ? qo0 - T.q_lo : qo0) + (uint32_t)r.s1;
                            sgm.nibabs = (staged ? (so0 - T.s_lo) * 2u : so0 * 2u) + (uint32_t)r.s1;
                            sm.segs[idx] = sgm;
                        } else {
                            TileSink sink; sink.P = &P; sink.sm = sm; sink.staged = false; sink.qabs0 = qo0; sink.nibabs0 = so0 * 2u;
                            sink.seq_read = P.b.seq + so0; sink.qual_read = P.b.qual + qo0; sink.errs = 0;
                            sink.push(pos, r.m, r.s1);                                // list full: exact serial path
                            if (sink.errs) atomic_or(P.err, sink.errs);
                        }
                        atomic_min(&sm.ctrl[C_TMIN], pos); atomic_max(&sm.ctrl[C_TMAX], pos + r.m);
                    }
                } else {
                    const int k = atomic_add(&sm.ctrl[C_NCPX], 1);
                    clist[k] = (uint16_t)rr;
                    if (do_pile && pos >= 0) {   // bound where it can pile up: trimming never leaves the input span
                        atomic_min(&sm.ctrl[C_TMIN], pos); atomic_max(&sm.ctrl[C_TMAX], pos + ref_len_of(cig, nc));
                    }
                }
            }
        }
        AMP_SYNC(); AMP_TICK(1);
        // ---- W: window decision (uniform) -----------------------------------------------------------
        int ncpx = sm.ctrl[C_NCPX];
        int nseg0 = sm.ctrl[C_NSEG]; if (nseg0 > P.maxseg) nseg0 = P.maxseg;
        // A handful of queued reads would keep one warp on the slow generic path for the whole tile: collect them
        // and run them together at the end of the CTA (unstaged, but with every lane busy).  Tiles that are mostly
        // generic (indel-rich data) are processed in place, where their rows are staged.
#if AMP_DEFER_MAX > 0
        if (ncpx > 0 && ncpx <= AMP_DEFER_MAX && ndef + ncpx <= AMP_DLIST_CAP) {
            AMP_FOR_THREADS(tid, nthreads) {
                if (tid < ncpx) dlist[ndef + tid] = (uint32_t)(T.t0 - P.b.first) + clist[tid];
            }
            ndef += ncpx; ncpx = 0;
        }
#endif
        if (do_pile) {
            const int tmin = sm.ctrl[C_TMIN], tmax = sm.ctrl[C_TMAX];
            if (tmax >= 0 && (wbase < 0 || tmin < wbase || tmax > wbase + P.wt)) {
                if (wbase >= 0) {
                    AMP_FOR_THREADS(tid, nthreads) { flush_tile(P, sm.cnt, wbase, tid, nthreads, true); }
                    AMP_SYNC();
                }
                wbase = tmin & ~31;
            }
        }
        AMP_TICK(2);
        // ---- T1 + C: queued reads take the generic path (their runs go to the tail of the list) while the other
        // warps already count the runs planned in T0.
        AMP_FOR_THREADS(tid, nthreads) {
            for (int k = tid; k < ncpx; k += nthreads) read_generic<DIRECT>(P, sm, T, (int)clist[k], DIRECT && ncpx > AMP_DIRECT_MIN, wbase);
        }
        if (do_pile) {
            AMP_FOR_THREADS(tid, nthreads) { count_runs(P, sm, 0, nseg0, wbase, tid, nthreads, (ncpx + 31) >> 5); }
        }
        AMP_SYNC(); AMP_TICK(3);
        if (do_pile && ncpx > 0) {
            int nseg = sm.ctrl[C_NSEG]; if (nseg > P.maxseg) nseg = P.maxseg;
            if (nseg > nseg0) {
                AMP_FOR_THREADS(tid, nthreads) { count_runs(P, sm, nseg0, nseg, wbase, tid, nthreads, 0); }
            }
            AMP_SYNC();
        }
    }
#if defined(__CUDA_ARCH__) && defined(AMP_PHASE_TIMING)
    if (threadIdx.x == 0 && P.phase_cycles) for (int k = 0; k < 4; ++k) P.phase_cycles[(size_t)block * 4 + k] = tacc[k];
#endif
    // ---- D: deferred reads of the whole CTA, generic path straight from global memory ----------------------------
#if AMP_DEFER_MAX > 0
    if (ndef > 0) {
        TileCtx T;
        T.t0 = P.b.first; T.nreads = 0; T.q_lo = T.q_hi = T.s_lo = T.s_hi = 0; T.do_trim = do_trim; T.do_pile = do_pile;
        T.q_glo = P.b.qual_off[P.b.first]; T.q_ghi = P.b.qual_off[P.b.first + P.b.n];
        AMP_FOR_THREADS(tid, nthreads) {
            if (tid == 0) { sm.ctrl[C_NSEG] = 0; sm.ctrl[C_TMIN] = 0x7FFFFFFF; sm.ctrl[C_TMAX] = -1; }
        }
        AMP_SYNC();
        AMP_FOR_THREADS(tid, nthreads) {
            for (int k = tid; k < ndef; k += nthreads) read_generic<DIRECT>(P, sm, T, (int)dlist[k], false, wbase);
        }
        AMP_SYNC();
        if (do_pile) {
            int nseg = sm.ctrl[C_NSEG]; if (nseg > P.maxseg) nseg = P.maxseg;
            const int tmin = sm.ctrl[C_TMIN], tmax = sm.ctrl[C_TMAX];
            if (tmax >= 0 && (wbase < 0 || tmin < wbase || tmax > wbase + P.wt)) {
                if (wbase >= 0) {
                    AMP_FOR_THREADS(tid, nthreads) { flush_tile(P, sm.cnt, wbase, tid, nthreads, true); }
                    AMP_SYNC();
                }
                wbase = tmin & ~31;
            }
            AMP_FOR_THREADS(tid, nthreads) { count_runs(P, sm, 0, nseg, wbase, tid, nthreads, 0); }
            AMP_SYNC();
        }
    }
#endif
    if (do_pile && wbase >= 0) {
        AMP_FOR_THREADS(tid, nthreads) { flush_tile(P, sm.cnt, wbase, tid, nthreads, false); }
    }
}

// ---------------------------------------------------------------------------------------------------
// Calling (AmpliPy.py:756-771, 919-951): the serial form, one thread per (sample, position); the CPU emulation's reference
// for the kernel's body (amp_call.cuh).
// ---------------------------------------------------------------------------------------------------
struct CallParams {
    int L, Lpad, n_samples;
    const int* counts;                 // [n_samples][6][Lpad]
    const InsSlot* slots;              // insertion table (heads[] / next chains: InsTable, linked by ins_table_add)
    const int* slot_entry;             // slot -> dense allele index k (amp_ins_export order)
    const unsigned char* arena;
    const int* heads;                  // [n_samples * Lpad] slot index of the first insertion allele, -1 = none
    const unsigned char* ref_seq;      // raw FASTA characters: [L], or [n_samples][ref_stride] when samples have references of their own
    long long ref_stride;              // 0: one reference for every sample
    int min_depth_consensus; double min_freq_consensus;
    int min_depth_variants; double min_freq_variants;
    // outputs
    int* depth;                        // [S*L] total depth incl. insertion alleles (767)
    int* top_id;                       // [S*L] allele id of the top allele: 0..5 = ACGTN-, 6 + k = insertion allele k, -1 none
    int* top_count;                    // [S*L]
    unsigned char* pos_flags;          // [S*L] bit0 consensus passes (928), bit1 variant record emitted (940), bit2 GT has ref (948)
    int* ref_count;                    // [S*L]
    double* fixed_freq;                // [S*L*6] count/total (float64, IEEE division)
    int* fixed_rank;                   // [S*L*6] index in the reference's sorted allele list, -1 if count == 0
    unsigned char* alt_mask;           // [S*L] bit ch: fixed symbol ch is an ALT allele (938)
    double* ins_freq;                  // [n_alleles] per insertion allele, dense index k
    int* ins_rank;                     // [n_alleles]
    unsigned char* ins_alt;            // [n_alleles]
};

// python string order between two allele symbols (fixed symbols are 1-char strings)
struct Sym { const unsigned char* p; int len; };
AMP_HD int sym_cmp(const Sym& a, const Sym& b) {
    int m = a.len < b.len ? a.len : b.len;
    for (int i = 0; i < m; ++i) { if (a.p[i] != b.p[i]) return a.p[i] < b.p[i] ? -1 : 1; }
    return a.len - b.len;
}
AMP_HD bool allele_greater(int ca, const Sym& a, int cb, const Sym& b) {   // (count, freq, symbol) descending
    if (ca != cb) return ca > cb;
    return sym_cmp(a, b) > 0;
}
AMP_HD Sym slot_sym(const CallParams& P, int slot) {
    const unsigned char* rec = P.arena + (P.slots[slot].key & 0xFFFFFFFFFFULL) * 8;
    Sym s; s.p = rec + 8; s.len = (int)((const unsigned int*)rec)[1]; return s;
}

// The insertion alleles of one position, either walked through the linked list on every use or (the normal case)
// copied once into per-thread arrays: the O(k^2) allele ordering then costs k dependent global loads instead of k^2.
struct ChainLinked {
    const CallParams* P; int head;
    AMP_HD int first() const { return head; }
    AMP_HD int next(int it) const { return P->slots[it].next; }
    AMP_HD bool valid(int it) const { return it >= 0; }
    AMP_HD int count(int it) const { return P->slots[it].count; }
    AMP_HD Sym sym(int it) const { return slot_sym(*P, it); }
    AMP_HD int slot(int it) const { return it; }
};
#define AMP_CHAIN_MAX 24
struct ChainCached {
    int n; int slot_[AMP_CHAIN_MAX], cnt_[AMP_CHAIN_MAX]; Sym sym_[AMP_CHAIN_MAX];
    AMP_HD int first() const { return 0; }
    AMP_HD int next(int it) const { return it + 1; }
    AMP_HD bool valid(int it) const { return it < n; }
    AMP_HD int count(int it) const { return cnt_[it]; }
    AMP_HD Sym sym(int it) const { return sym_[it]; }
    AMP_HD int slot(int it) const { return slot_[it]; }
};

template <class Chain>
AMP_HD void call_position_impl(const CallParams& P, const unsigned char* fixed_syms, long long gp, int p, const int* c, long long total,
                               const Chain& ch_) {
    P.depth[gp] = (int)total;
    int best_id = -1, best_c = 0; Sym best_s; best_s.p = fixed_syms; best_s.len = 0;
    int refc = 0; double reff = 0.0; unsigned alt = 0; int n_alt = 0;
    const unsigned char refsym = P.ref_seq[(size_t)(gp / P.L) * (size_t)P.ref_stride + p];
    for (int ch = 0; ch < AMP_NCH; ++ch) {
        double f = total ? (double)c[ch] / (double)total : 0.0;
        P.fixed_freq[gp * AMP_NCH + ch] = f;
        int rank = -1;
        if (c[ch]) {
            Sym me; me.p = fixed_syms + ch; me.len = 1;
            rank = 0;
            for (int o = 0; o < AMP_NCH; ++o) if (o != ch && c[o]) { Sym os; os.p = fixed_syms + o; os.len = 1; if (allele_greater(c[o], os, c[ch], me)) ++rank; }
            for (int t = ch_.first(); ch_.valid(t); t = ch_.next(t)) if (ch_.count(t) && allele_greater(ch_.count(t), ch_.sym(t), c[ch], me)) ++rank;
            if (best_id < 0 || allele_greater(c[ch], me, best_c, best_s)) { best_id = ch; best_c = c[ch]; best_s = me; }
            if (fixed_syms[ch] == refsym) { refc = c[ch]; reff = f; }                  // 936-937
            else if (f >= P.min_freq_variants) { alt |= 1u << ch; ++n_alt; }           // 938-939
        }
        P.fixed_rank[gp * AMP_NCH + ch] = rank;
    }
    for (int s = ch_.first(); ch_.valid(s); s = ch_.next(s)) {
        const int cs = ch_.count(s);
        if (!cs) continue;
        const Sym me = ch_.sym(s);
        const double f = (double)cs / (double)total;
        int rank = 0;
        for (int o = 0; o < AMP_NCH; ++o) if (c[o]) { Sym os; os.p = fixed_syms + o; os.len = 1; if (allele_greater(c[o], os, cs, me)) ++rank; }
        for (int t = ch_.first(); ch_.valid(t); t = ch_.next(t)) if (t != s && ch_.count(t) && allele_greater(ch_.count(t), ch_.sym(t), cs, me)) ++rank;
        const int kk = P.slot_entry[ch_.slot(s)];
        P.ins_freq[kk] = f; P.ins_rank[kk] = rank;
        if (best_id < 0 || allele_greater(cs, me, best_c, best_s)) { best_id = 6 + kk; best_c = cs; best_s = me; }
        // an insertion key can never equal the 1-character reference symbol except a 1-char key, which
        // the pileup already routed to the fixed channels
        unsigned char is_alt = 0;
        if (me.len == 1 && me.p[0] == refsym) { refc = cs; reff = f; }
        else if (f >= P.min_freq_variants) is_alt = 1;
        P.ins_alt[kk] = is_alt; n_alt += is_alt;
    }
    P.top_id[gp] = best_id; P.top_count[gp] = best_c;
    unsigned char fl = 0;
    if (best_id >= 0) {
        const double bf = (double)best_c / (double)total;
        if (best_c >= P.min_depth_consensus && bf >= P.min_freq_consensus) fl |= 1;     // 928
    }
    if (total > 0 && total >= P.min_depth_variants && n_alt != 0) {                    // 940
        fl |= 2;
        if (refc >= P.min_depth_variants && reff >= P.min_freq_variants) fl |= 4;      // 948
    }
    P.pos_flags[gp] = fl; P.ref_count[gp] = refc; P.alt_mask[gp] = (unsigned char)alt;
}

AMP_HD void call_position(const CallParams& P, const unsigned char* fixed_syms, long long gp) {
    const int sample = (int)(gp / P.L), p = (int)(gp - (long long)sample * P.L);
    const int* cnt = P.counts + (size_t)sample * AMP_NCH * P.Lpad;
    int c[AMP_NCH]; long long total = 0;
    for (int ch = 0; ch < AMP_NCH; ++ch) { c[ch] = cnt[(size_t)ch * P.Lpad + p]; total += c[ch]; }
    const int head = P.heads[(size_t)sample * P.Lpad + p];
    ChainCached cc; cc.n = 0;
    int k = 0;
    for (int s = head; s >= 0; s = P.slots[s].next, ++k) {
        const int cs = P.slots[s].count;
        total += cs;
        if (k < AMP_CHAIN_MAX) { cc.slot_[k] = s; cc.cnt_[k] = cs; }
    }
    if (k <= AMP_CHAIN_MAX) {
        cc.n = k;
        for (int j = 0; j < k; ++j) cc.sym_[j] = slot_sym(P, cc.slot_[j]);
        call_position_impl(P, fixed_syms, gp, p, c, total, cc);
    } else {
        ChainLinked cl; cl.P = &P; cl.head = head;
        call_position_impl(P, fixed_syms, gp, p, c, total, cl);
    }
}

}  // namespace amp
