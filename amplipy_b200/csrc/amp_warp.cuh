// amp_warp.cuh -- warp-autonomous fused trim + pileup kernel for short-read batches (sm_100a).
//
// One CTA per SM owns a contiguous chunk of the (coordinate-sorted) reads and one privatised count tile over the
// reference window of that chunk, indexed directly by the BAM base nibble (18 rows x WT: rows 1,2,4,8,15 = A,C,G,T,N;
// row 16 = sink for masked bases, never read; row 17 = '-'; any other row only raises the KeyError flag at the flush).  The warps are
// autonomous: no block barrier between set-up and the final flush.
//
// Batch warps loop over batches of up to 32 consecutive reads, software-pipelined over the batches:
//   A  lane per read : [H][S]M[(I|D)M][S][H] classification (Shape5, amp_core.cuh) and the closed form of the two primer clips (trim_read,
//                      AmpliPy.py:450-558) from metadata / CIGAR words loaded one batch ahead; lane 0 starts one bulk async
//                      copy (cp.async.bulk, completion on an mbarrier) per array that drops the batch's contiguous quality /
//                      sequence byte ranges into the warp's staging buffers.
//   B1 lane per read : sliding-window search (566-587 / 628-649) over aligned words of the row: eight windows per step
//                      (dp4a against -4*minq), one "some window fails" bit per block, the first (forward) / last (reverse)
//                      failing block resolved exactly; quality clip + write gate (589-686, 910); trim outputs.
//   B2 pileup        : (update_base_counts, 718 + 752-753) the 8-base chunks of the batch's aligned runs are dealt out
//                      evenly over the 32 lanes; per chunk a SIMD byte compare q >= minq, per base one byte permute (row
//                      offset), one select (sink row for masked bases), one add, one shared-memory atomic.
//   G  every read the closed form declines (three or more alignment ops, odd clips, equal neighbours) goes to the CTA's list.
//      When the batches are done the generic-capable warps work through it (AMP7_DWARPS > 0: that many warps do nothing
//      else from the start; measured no better): rows staged with one bulk copy per lane, the loop-for-loop generic path
//      lane per read (trim_read + plan_read of amp_core.cuh on CIGAR rows in shared memory), runs counted with the
//      balanced chunk loop.
//
// tests/emu runs this very source on the CPU with every CUDA thread as a fiber (warp collectives, barriers and spin-waits
// are rendezvous / yield points of a deterministic scheduler).
#pragma once
#include <string.h>

#include "amp_kernels.cuh"

namespace amp {

// ---- warp / CTA primitives: hardware on the device, fibers in tests/emu -------------------------------------------
#if defined(__CUDA_ARCH__)
#define AMP_WD __device__ __forceinline__
#define AMP_WD_COLD __device__ __noinline__            // rarely executed: kept out of the hot loops' instruction footprint
AMP_WD int c_tid() { return (int)threadIdx.x; }
AMP_WD int c_nthreads() { return (int)blockDim.x; }
AMP_WD int c_block() { return (int)blockIdx.x; }
AMP_WD int w_shfl(int v, int src) { return __shfl_sync(0xFFFFFFFFu, v, src); }
AMP_WD unsigned w_ballot(bool p) { return __ballot_sync(0xFFFFFFFFu, p); }
AMP_WD int w_add(int v) { return __reduce_add_sync(0xFFFFFFFFu, v); }
AMP_WD void w_sync() { __syncwarp(); }
AMP_WD void c_sync() { __syncthreads(); }
AMP_WD void c_yield() { __nanosleep(200); }                        // polite spin-wait
AMP_WD int ld_vol(const int* p) { return *(const volatile int*)p; }
AMP_WD void st_vol(int* p, int v) { *(volatile int*)p = v; }
AMP_WD uint32_t ld_cg_u32(const uint32_t* p) { return __ldcg(p); }  // L2: entries written by another warp of the CTA
AMP_WD void st_cg_u32(uint32_t* p, uint32_t v) { __stcg(p, v); }
AMP_WD void fence_block() { __threadfence_block(); }
AMP_WD int popc32(unsigned x) { return __popc(x); }
AMP_WD unsigned byte_perm2(unsigned x, unsigned sel) { return __byte_perm(x, 0u, sel); }
// prmt.b32 with the selector's replicate-sign bit honoured: nibble 8 + k = byte k's top bit over the whole byte
AMP_WD unsigned prmt_sx(unsigned a, unsigned b, unsigned sel) {
    unsigned r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}
AMP_WD uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
AMP_WD void mbar_init(unsigned long long* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// start the bulk copies of one batch: expect `total` bytes on the barrier, then up to two copies
AMP_WD void bulk_expect(unsigned long long* bar, uint32_t total) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic-proxy accesses of the buffers are done
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(total) : "memory");
}
AMP_WD void bulk_copy(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
// pull [src, src + bytes) towards L2 (bytes a multiple of 16); purely a hint
AMP_WD void bulk_prefetch_l2(const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
AMP_WD void bulk_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok)
                     : "r"(smem_addr(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}
#else
#define AMP_WD inline
#define AMP_WD_COLD inline
// implemented by the fiber runtime in tests/emu/amp_emu.cpp
int c_tid(); int c_nthreads(); int c_block();
int w_shfl(int v, int src); unsigned w_ballot(bool p); int w_add(int v);
void w_sync(); void c_sync(); void c_yield();
AMP_WD int ld_vol(const int* p) { return *p; }
AMP_WD void st_vol(int* p, int v) { *p = v; }
AMP_WD uint32_t ld_cg_u32(const uint32_t* p) { return *p; }
AMP_WD void st_cg_u32(uint32_t* p, uint32_t v) { *p = v; }
AMP_WD void fence_block() {}
AMP_WD int popc32(unsigned x) { return __builtin_popcount(x); }
AMP_WD unsigned byte_perm2(unsigned x, unsigned sel) {
    unsigned r = 0;
    for (int i = 0; i < 4; ++i) { const unsigned k = (sel >> (4 * i)) & 7u; r |= (k < 4 ? (x >> (8 * k)) & 0xFFu : 0u) << (8 * i); }
    return r;
}
AMP_WD unsigned prmt_sx(unsigned a, unsigned b, unsigned sel) {
    unsigned r = 0;
    for (int i = 0; i < 4; ++i) {
        const unsigned n = (sel >> (4 * i)) & 15u, k = n & 7u;
        unsigned v = ((k < 4 ? a >> (8 * k) : b >> (8 * (k - 4))) & 0xFFu);
        if (n & 8u) v = (v & 0x80u) ? 0xFFu : 0u;
        r |= v << (8 * i);
    }
    return r;
}
AMP_WD void mbar_init(unsigned long long*) {}
AMP_WD void bulk_expect(unsigned long long*, uint32_t) {}
AMP_WD void bulk_copy(void* dst, const void* src, uint32_t bytes, unsigned long long*) { memcpy(dst, src, bytes); }
AMP_WD void bulk_wait(unsigned long long*, uint32_t) {}
AMP_WD void bulk_prefetch_l2(const void*, uint32_t) {}
static long long g_v7_stats[2];   // emulation only: reads finished on the cooperative path / reads sent to the generic path
#endif

// debug builds (-DAMP7_TIMING): per-warp cycle counters of the kernels' phases, summed over all warps into
// P.phase_cycles[base + k]; slot 7 of the local array holds the last time stamp
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
#define AMP7_T0(t) long long t[8] = {0, 0, 0, 0, 0, 0, 0, 0}; t[7] = clock64()
#define AMP7_TICK(t, k) do { const long long n_ = clock64(); (t)[k] += n_ - (t)[7]; (t)[7] = n_; } while (0)
#define AMP7_TDUMP(t, base) do { if ((threadIdx.x & 31) == 0 && P.phase_cycles) for (int k_ = 0; k_ < 7; ++k_) atomicAdd((unsigned long long*)&P.phase_cycles[(base) + k_], (unsigned long long)(t)[k_]); } while (0)
#else
#define AMP7_T0(t) long long* t = nullptr; (void)t
#define AMP7_TICK(t, k) ((void)0)
#define AMP7_TDUMP(t, base) ((void)0)
#endif

#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
#define AMP7_GT0() long long gt_ = clock64()
#define AMP7_GTICK(k) do { __syncwarp(__activemask()); const long long n_ = clock64(); if (P.phase_cycles && (__ffs(__activemask()) - 1) == (int)(threadIdx.x & 31)) atomicAdd((unsigned long long*)&P.phase_cycles[360 + (k)], (unsigned long long)(n_ - gt_)); gt_ = n_; } while (0)
#else
#define AMP7_GT0() ((void)0)
#define AMP7_GTICK(k) ((void)0)
#endif
#define AMP7_PRAGMA_(x) _Pragma(#x)
#define AMP7_UNROLL(n) AMP7_PRAGMA_(unroll n)
#ifndef AMP7_COUNT_UNROLL
#define AMP7_COUNT_UNROLL 1     // the count loop as it is: unrolled by the compiler it measured no faster and is twice the code
#endif

// ---- shared-memory layout ------------------------------------------------------------------------------------------
#ifndef AMP7_WARPS
#define AMP7_WARPS 20            // warps per CTA of the fast kernel (96 registers per thread; 20 warps + 2 generic-capable ones fill the 227 KB of shared memory)
#endif
#ifndef AMP7_GWARPS
#define AMP7_GWARPS 2            // warps that can run the generic phase (their extra shared memory must fit): the last ones
#endif
#ifndef AMP7_DWARPS
#define AMP7_DWARPS 0            // of those, warps that do nothing else (they work on the list while it is being filled)
#endif
#define AMP7_WT 512              // count tile width on the device (positions)
#define AMP7_SINK_ROW 16         // count tile rows: BAM nibble 0..15, row 16 = sink of masked bases (never read), then the '-' row
#define AMP7_SINK_SLACK 32       // the sink row is this much longer: masked bases of a run's last chunk land past the window's end
#define AMP7_PAD 16              // bytes in front of the staged data (phase B may address up to 3 nibbles before it)
#ifndef AMP7_QDATA
#define AMP7_QDATA 5120          // staged quality bytes per batch (32 x 150 + alignment)
#endif
#ifndef AMP7_SDATA
#define AMP7_SDATA 2560
#endif
#define AMP7_QSLACK 32           // the word-wise passes read up to 16 bytes past a run
#define AMP7_SSLACK 32
#define AMP7_QBUF (AMP7_PAD + AMP7_QDATA + AMP7_QSLACK)
#define AMP7_SBUF (AMP7_PAD + AMP7_SDATA + AMP7_SSLACK)
#ifndef AMP7_RUNCAP
#define AMP7_RUNCAP 80           // run descriptors per warp (generic path)
#endif
#define AMP7_QCAP 32             // generic-path reads per warp and round
#define AMP7_GSLOT_Q 192         // G phase: bytes per staged quality row slot
#define AMP7_GSLOT_S 96
#ifndef AMP7_GN
#define AMP7_GN 26               // reads per G phase (GN * GSLOT <= DATA)
#endif
#define AMP7_CROW 9              // generic path: CIGAR ops (+3) per shared-memory row; two rows per read (odd stride: no bank conflicts)
#define AMP7_GEXTRA_BYTES (AMP7_RUNCAP * 16 + AMP7_QCAP * 4 + 32 + AMP7_GN * 2 * AMP7_CROW * 4)   // generic phase: runs, queue, counters, CIGAR rows
#define AMP7_PSLICE 640          // positions of the two primer tables kept in shared memory, from the window base
#ifndef AMP7_EVCAP
#define AMP7_EVCAP 256           // insertion alleles of a CTA's reads wait here (three words each) until its batches are done
#endif
#ifndef AMP7_GLCAP
#define AMP7_GLCAP 512           // reads for the generic phase listed in shared memory (whatever does not fit: P.glist)
#endif
enum { C7_TMIN = 0, C7_NEXT = 1, C7_NGEN = 2, C7_GNEXT = 3, C7_FASTDONE = 4, C7_NEV = 5, C7_EVDONE = 6, C7_PTAB = 16, C7_EV = C7_PTAB + 2 * AMP7_PSLICE,
       C7_GL = C7_EV + 3 * AMP7_EVCAP, C7_WORDS = C7_GL + AMP7_GLCAP };

AMP_HD int del_row_off(int wt) { return (AMP7_SINK_ROW + 1) * wt + AMP7_SINK_SLACK; }      // first element of the '-' row
AMP_HD size_t tile_bytes_v7(int wt) { return ((size_t)(AMP7_SINK_ROW + 2) * wt + AMP7_SINK_SLACK) * 4; }
AMP_HD size_t smem_bytes_v9(int wt, int warps, int gwarps);   // below

// One aligned run of the count pass, fully decoded by its owner lane so that switching runs inside the chunk loop is cheap:
//   qoff / soff = byte offset, from the start of the count tile, of the aligned quality / sequence word of chunk 0
//   toff = the same of the tile element (row 0) of chunk 0's first base
//   k = quality funnel shift (bits) | sequence funnel shift << 8 | chunks << 16 | odd first nibble << 24
//   mka/mkb = byte masks of the last chunk's bases 0,2,4,6 / 1,3,5,7, mfa/mfb = of the first chunk's (phi bases in front)
// Everything a lane needs when it moves on to the next run is a plain copy of these words (the switch sits in the count loop and
// runs in almost every iteration for some lane of the warp, so each of its instructions counts like one of the loop body).
struct Par4 { unsigned qoff, soff, toff, k, mka, mkb, mfa, mfb; };
AMP_WD Par4 make_par(unsigned qbase, unsigned sbase, int a0, int n0, int m, int phi, int z) {   // a0 / n0 / z: of the first of the m bases (incl. phi in front)
    Par4 p;
    const int sb = n0 >> 1, nch = (m + 7) >> 3;
    p.qoff = qbase + (unsigned)(a0 & ~3);
    p.soff = sbase + (unsigned)(sb & ~3);
    p.toff = 4u * (unsigned)z;
    p.k = (unsigned)((a0 & 3) << 3) | ((unsigned)((sb & 3) << 3) << 8) | ((unsigned)nch << 16) | ((unsigned)(n0 & 1) << 24);
    const int left = m - 8 * (nch - 1);              // bases of the last chunk, 1 .. 8
    const unsigned mk0 = left >= 4 ? 0xFFFFFFFFu : (1u << (8 * left)) - 1u;
    const unsigned mk1 = left >= 8 ? 0xFFFFFFFFu : (left > 4 ? (1u << (8 * (left - 4))) - 1u : 0u);
    const unsigned mf0 = phi >= 4 ? 0u : 0xFFFFFFFFu << (8 * phi);
    const unsigned mf1 = phi > 4 ? 0xFFFFFFFFu << (8 * (phi - 4)) : 0xFFFFFFFFu;
    p.mka = prmt_sx(mk0, mk1, 0x6420u); p.mkb = prmt_sx(mk0, mk1, 0x7531u);
    p.mfa = prmt_sx(mf0, mf1, 0x6420u); p.mfb = prmt_sx(mf0, mf1, 0x7531u);
    return p;
}
struct V7Cfg { int wt, batch_reads; };
inline V7Cfg pick_v7_cfg(long long n, long long sum_qual, int sm_count) {
    (void)sm_count;
    V7Cfg t;
    t.wt = AMP7_WT;
    const double avg_len = n ? (double)sum_qual / (double)n : 150.0;
    int br = (int)((AMP7_QDATA - 16) / (avg_len * 1.02 + 1.0));
    t.batch_reads = br < 1 ? 1 : (br > 32 ? 32 : br);
    return t;
}

// fast kernel: per-warp staging buffers, the per-run parameters of the count pass, and the bulk-copy barrier
#define AMP7_FAST_BYTES (AMP7_QBUF + AMP7_SBUF + 32 * 32 + 64 + 16)
struct FastMem { uint8_t* qbuf; uint8_t* sbuf; Par4* par; uint16_t* own; unsigned long long* bar; };
AMP_HD size_t smem_bytes_fast(int wt, int warps) { return tile_bytes_v7(wt) + C7_WORDS * 4 + (size_t)warps * AMP7_FAST_BYTES; }
AMP_HD FastMem carve_fast(unsigned char* base, int wt, int w) {
    unsigned char* b = base + tile_bytes_v7(wt) + C7_WORDS * 4 + (size_t)w * AMP7_FAST_BYTES;
    FastMem m;
    m.qbuf = b; b += AMP7_QBUF;
    m.sbuf = b; b += AMP7_SBUF;
    m.par = (Par4*)b; b += 32 * 32;
    m.own = (uint16_t*)b; b += 64;
    m.bar = (unsigned long long*)b;
    return m;
}

struct WarpMem7 {
    uint8_t* qbuf; uint8_t* sbuf; Seg* runs; uint32_t* queue; int* ctr; unsigned long long* bar; uint32_t* cig;
    Par4* par; uint16_t* own; int* ctrl;
};
AMP_HD size_t smem_bytes_v9(int wt, int warps, int gwarps) {
    return tile_bytes_v7(wt) + C7_WORDS * 4 + (size_t)warps * AMP7_FAST_BYTES + (size_t)gwarps * AMP7_GEXTRA_BYTES;
}
// generic phase: the warp's fast-part buffers + its extra block behind all fast-part blocks
AMP_HD WarpMem7 carve_warp7(unsigned char* base, int wt, int warps, int gwarps, int g) {   // g-th generic-capable warp = warp warps - gwarps + g
    const FastMem f = carve_fast(base, wt, warps - gwarps + g);
    unsigned char* b = base + tile_bytes_v7(wt) + C7_WORDS * 4 + (size_t)warps * AMP7_FAST_BYTES + (size_t)g * AMP7_GEXTRA_BYTES;
    WarpMem7 m;
    m.qbuf = f.qbuf; m.sbuf = f.sbuf; m.par = f.par; m.own = f.own; m.bar = f.bar;
    m.runs = (Seg*)b; b += AMP7_RUNCAP * 16;
    m.queue = (uint32_t*)b; b += AMP7_QCAP * 4;
    m.ctr = (int*)b; b += 32;
    m.cig = (uint32_t*)b;
    m.ctrl = (int*)(base + tile_bytes_v7(wt));
    return m;
}

// channel of a nibble row, -1 = not a countable base
AMP_HD int row_channel(int row) { return nib_channel((uint32_t)row); }

// tile -> global count matrix; rows that are no base only raise the KeyError flag (AmpliPy.py:753).  A thread per position: all
// its loads are independent (one round trip to shared memory instead of one per row).
AMP_HD void flush_tile7(const KParams& P, const int* cnt, int wbase, int tid, int nthreads) {
    const int wt = P.wt;
    const int* del = cnt + del_row_off(wt);
    for (int w = tid; w < wt; w += nthreads) {
        const int a = cnt[1 * wt + w], c = cnt[2 * wt + w], g = cnt[4 * wt + w], t = cnt[8 * wt + w], n = cnt[15 * wt + w], d = del[w];
        int bad = cnt[w] | cnt[3 * wt + w];
        for (int row = 5; row < 15; ++row) if (row != 8) bad |= cnt[row * wt + w];
        int* out = P.counts + wbase + w;
        if (a) atomic_add(out, a);
        if (c) atomic_add(out + (size_t)1 * P.Lpad, c);
        if (g) atomic_add(out + (size_t)2 * P.Lpad, g);
        if (t) atomic_add(out + (size_t)3 * P.Lpad, t);
        if (n) atomic_add(out + (size_t)4 * P.Lpad, n);
        if (d) atomic_add(out + (size_t)5 * P.Lpad, d);
        if (bad) atomic_or(P.err, AMP_E_BASE);
    }
}

// An insertion allele of a read: straight into the table, or (the CTA's list has room) parked until the CTA's batches are
// done, when all of them are added with one thread each -- inside the per-read code an add would run with one lane active.
AMP_HD void ins_commit(const KParams& P, const uint8_t* seq_read, int pos, int b, int n) {
    if (n == 1) {   // one-character key == that base's own dict entry (AmpliPy.py:745-746)
        const int ch = nib_channel(nib_at(seq_read, (uint32_t)b));
        if (ch >= 0) { atomic_add(&P.counts[(size_t)ch * P.Lpad + pos], 1); return; }
    }
    TileSink::Text t; t.seq = seq_read; t.b = b;
    ins_table_add(P.tab, P.gpos_base + pos, n, t, 1);
}
AMP_WD_COLD void ins_defer(const KParams& P, int* ctrl, uint32_t so0, int pos, int b, int n) {   // so0: the read's offset in P.b.seq
    if (b < 65536 && n > 0 && n < 65536) {
        const int idx = atomic_add(&ctrl[C7_NEV], 1);
        if (idx < AMP7_EVCAP) {      // the third word (never 0) is written last: it tells a draining warp that the entry is complete
            int* e = ctrl + C7_EV + 3 * idx;
            e[0] = pos; e[1] = (int)so0;
            fence_block();
            st_vol(&e[2], (int)((uint32_t)b | ((uint32_t)n << 16)));
            return;
        }
    }
    ins_commit(P, P.b.seq + so0, pos, b, n);
}
// Add parked alleles to the table, up to 32 at a time (a lane each), until none is left: called by warps that have run out
// of batches while the others still append, and by every warp once all of them are done.
AMP_WD void ins_drain(const KParams& P, int* ctrl, int lane) {
    for (;;) {
        int at = -1, n = 0;
        if (lane == 0) {
            for (;;) {
                const int done = ld_vol(&ctrl[C7_EVDONE]);
                int have = ld_vol(&ctrl[C7_NEV]); if (have > AMP7_EVCAP) have = AMP7_EVCAP;
                if (have <= done) break;
                n = have - done < 32 ? have - done : 32;
                if (atomic_cas(&ctrl[C7_EVDONE], done, done + n) == done) { at = done; break; }
            }
        }
        at = w_shfl(at, 0); n = w_shfl(n, 0);
        if (at < 0) return;
        if (lane < n) {
            int* e = ctrl + C7_EV + 3 * (at + lane);
            int w;
            while ((w = ld_vol(&e[2])) == 0) c_yield();            // reserved but not yet written
            fence_block();
            ins_commit(P, P.b.seq + (uint32_t)ld_vol(&e[1]), ld_vol(&e[0]), (int)((uint32_t)w & 0xFFFFu), (int)((uint32_t)w >> 16));
        }
        w_sync();
    }
}

// ---- lane-per-read passes over a staged read ---------------------------------------------------------------------------
// `buf + a0` = first aligned quality byte (any alignment), m aligned bases, window width 4.  Both passes walk aligned
// 4-byte words of the staging buffer and funnel-shift them to read-relative words; they read at most 16 bytes past the run.

// Pileup of one aligned run (update_base_counts, AmpliPy.py:718 + 752-753) inside the count tile: quality byte t at
// qbuf[a0 + t], base t = nibble n0 + t of sbuf, tile position tp0 + t, t in [0, m); this call covers the 8-base chunks
// [c_lo, c_hi).  Per chunk: two quality words -> SIMD byte compare q >= minq (bit 7 of each byte), spread by two
// sign-replicating byte permutes into byte masks in the order of the base words; one sequence word split into pre-scaled
// high / low nibbles (bases 0,2,4,6 / 1,3,5,7), masked bases replaced by the sink row's code with one logic op per word;
// then per base one byte permute (row offset), one add, one shared-memory atomic.  Lanes of a warp that work on reads
// with the same start hit the same address and are merged by the hardware (ATOMS.POPC.INC).
//
// The chunks of all runs of a batch are dealt out evenly: this lane walks chunks [g0, g1) of their concatenation,
// starting at chunk c0 of run rr0 (par[] lists the runs) and moving on to the next run inside the loop, so every lane of the
// warp executes the same number of iterations.
template <int WT>
AMP_WD void count_chunks_v9(int* cnt, int wt, const Par4* par, int rr0, int c0, int g0, int g1, unsigned minq4) {
    const char* base = (const char*)cnt;
    const Par4* pp = par + rr0;
    const Par4 p0 = *pp;
    int rem = (int)((p0.k >> 16) & 0xFFu) - c0;              // chunks of the current run still to do (>= 1)
    const uint32_t* A = (const uint32_t*)(base + p0.qoff) + 2 * c0;
    const uint32_t* S = (const uint32_t*)(base + p0.soff) + c0;
    unsigned sh = p0.k, ssh = p0.k >> 8;                     // (funnel shifts use the low five bits)
    bool odd = (p0.k >> 24) != 0;
    unsigned qa = A[0], sa = S[1], x = funnel_r(S[0], sa, ssh);
    int* tl = (int*)(base + p0.toff) + 8 * c0;
    unsigned mka = p0.mka, mkb = p0.mkb, ma = c0 == 0 ? p0.mfa : 0xFFFFFFFFu, mb = c0 == 0 ? p0.mfb : 0xFFFFFFFFu;
    const unsigned nminq4 = 0u - minq4;
#if defined(__CUDA_ARCH__) && defined(AMP7_COUNT_UNROLL)
    AMP7_UNROLL(AMP7_COUNT_UNROLL)
#endif
    for (int g = g0; g < g1; ++g) {
        if (rem == 0) {                                      // next run, from its chunk 0
            const Par4 pr = *++pp;
            rem = (int)((pr.k >> 16) & 0xFFu);
            A = (const uint32_t*)(base + pr.qoff); S = (const uint32_t*)(base + pr.soff);
            sh = pr.k; ssh = pr.k >> 8; odd = (pr.k >> 24) != 0;
            qa = A[0]; sa = S[1]; x = funnel_r(S[0], sa, ssh);
            tl = (int*)(base + pr.toff);
            mka = pr.mka; mkb = pr.mkb; ma = pr.mfa; mb = pr.mfb;
        }
        const unsigned q1 = A[1], q2 = A[2];
        const unsigned v0 = funnel_r(qa, q1, sh), v1 = funnel_r(q1, q2, sh);
        qa = q2; A += 2;
        const unsigned s2 = S[2];
        const unsigned xn = funnel_r(sa, s2, ssh);          // sequence word of the next chunk
        sa = s2; S += 1;
        // q >= minq per byte (exact for every byte value, minq <= 127): bit 7 of each byte
        const unsigned t0 = ((v0 | 0x80808080u) + nminq4) | v0;
        const unsigned t1 = ((v1 | 0x80808080u) + nminq4) | v1;
        unsigned ka = prmt_sx(t0, t1, 0xECA8u) & ma, kb = prmt_sx(t0, t1, 0xFDB9u) & mb;   // 0xFF per passing base, in a / b order;
        ma = 0xFFFFFFFFu; mb = 0xFFFFFFFFu;                                               // bases in front of the run masked
        if (rem == 1) { ka &= mka; kb &= mkb; }             // bases past the run
        // nibbles scaled by 8, one per byte: E = bases at even nibble positions of x, O = odd ones
        const unsigned E = (x >> 1) & 0x78787878u, O = (x << 3) & 0x78787878u, En = (xn >> 1) & 0x78787878u;
        unsigned a = odd ? O : E;                            // bases 0, 2, 4, 6 of the chunk
        unsigned b = odd ? funnel_r(E, En, 8) : O;           // bases 1, 3, 5, 7
        x = xn;
        a = (a & ka) | (~ka & 0x80808080u);                  // masked bases: code 16 = the sink row
        b = (b & kb) | (~kb & 0x80808080u);
#define AMP7_BASE(ii, src, kbyte)                                                                                      \
        {                                                                                                              \
            if (WT == 512) {                                                                                           \
                const unsigned off = byte_perm2(src, 0x4404u | ((kbyte) << 4));       /* row * 2048 bytes */            \
                atomic_add((int*)((char*)tl + off) + (ii), 1);                                                         \
            } else {                                                                                                   \
                const unsigned row = ((src) >> (8 * (kbyte) + 3)) & 31u;                                               \
                atomic_add(tl + (int)row * wt + (ii), 1);                                                              \
            }                                                                                                          \
        }
        AMP7_BASE(0, a, 0) AMP7_BASE(1, b, 0) AMP7_BASE(2, a, 1) AMP7_BASE(3, b, 1)
        AMP7_BASE(4, a, 2) AMP7_BASE(5, b, 2) AMP7_BASE(6, a, 3) AMP7_BASE(7, b, 3)
#undef AMP7_BASE
        tl += 8; --rem;
    }
}

// Deal the chunks of up to 32 runs (one per lane; nchk = 0: this lane has none) out evenly over the warp and count them.
// Quality clipping leaves aligned runs of very different lengths; lane l takes chunks [l*q, (l+1)*q) of the concatenation.
// The chunk grid of run k starts phi = k & 7 bases in front of the run (those bases are masked): in coordinate-sorted
// amplicon data most runs of a batch start at the same position, and lanes that are at different chunks of such runs would
// otherwise all fall into the same four banks of the tile (phi <= w0: never in front of the tile).
template <int WT>
AMP_WD void count_runs_balanced(int* cnt, int wt, const uint8_t* qbuf, const uint8_t* sbuf, Par4* par, uint16_t* own, int lane, bool has,
                                int a0, int n0, int m, int w0, unsigned minq4) {
    const unsigned hmask = w_ballot(has);                                      // the runs, in lane order
    if (!hmask) return;                                                        // uniform
    const int rank = popc32(hmask & ((1u << lane) - 1u)), phi = (rank & 7) < w0 ? (rank & 7) : (w0 > 0 ? w0 : 0);
    const int nchk = has ? (m + phi + 7) >> 3 : 0;
    int incl = nchk;
    for (int d = 1; d < 32; d <<= 1) { const int t = w_shfl(incl, lane - d); if (lane >= d) incl += t; }
    const int start = incl - nchk, total = w_shfl(incl, 31);
    const int q = (total + 31) >> 5;
    if (has) {
        par[rank] = make_par((unsigned)(qbuf - (const uint8_t*)cnt), (unsigned)(sbuf - (const uint8_t*)cnt), a0 - phi, n0 - phi, m + phi, phi, w0 - phi);
        const int l_hi = (start + nchk + q - 1) / q;
        for (int ll = (start + q - 1) / q; ll < l_hi && ll < 32; ++ll) own[ll] = (uint16_t)(rank | ((ll * q - start) << 8));   // lanes that start in this run, and at which chunk
    }
    w_sync();
    const int g0 = lane * q, g1 = g0 + q < total ? g0 + q : total;
    if (g0 < g1) { const int o = own[lane]; count_chunks_v9<WT>(cnt, wt, par, o & 0xFF, o >> 8, g0, g1, minq4); }
    w_sync();                                                                  // par / own may be rewritten
}

// ---- generic path inside a warp (same logic as TileSink / read_generic, warp-private run list) --------------------
struct WarpSink7 {
    const KParams* P; WarpMem7 wm;
    uint32_t qabs0, nibabs0, so0; bool staged;   // so0: the read's offset in P.b.seq
    const uint8_t* seq_read; const uint8_t* qual_read;
    unsigned int errs;
    AMP_HD void push(int rpos, int len_kind, int q) {
        const int idx = atomic_add(&wm.ctr[0], 1);
        if (idx < AMP7_RUNCAP) {
            Seg s; s.rpos = rpos; s.len = len_kind | (staged ? 0x40000000 : 0); s.qabs = qabs0 + (uint32_t)q; s.nibabs = nibabs0 + (uint32_t)q;
            wm.runs[idx] = s;
        } else {   // list full: exact serial path into the global matrix
            const int n = len_kind & 0x3FFFFFFF;
            if (len_kind < 0) { for (int j = 0; j < n; ++j) atomic_add(&P->counts[(size_t)5 * P->Lpad + rpos + j], 1); }
            else for (int j = 0; j < n; ++j) {
                if (qual_read[q + j] < P->tp.min_quality) continue;
                const int ch = nib_channel(nib_at(seq_read, (uint32_t)(q + j)));
                if (ch < 0) { errs |= AMP_E_BASE; continue; }
                atomic_add(&P->counts[(size_t)ch * P->Lpad + rpos + j], 1);
            }
        }
    }
    AMP_HD void match(int rpos, int q, int n) { push(rpos, n, q); }
    AMP_HD void del(int rpos, int n, int /*qa*/) { push(rpos, (int)(0x80000000u | (unsigned)n), 0); }
    AMP_WD void ins(int pos, int b, int n, int /*q0*/) { ins_defer(*P, wm.ctrl, so0, pos, b, n); }
};

// one base outside the tile (or of an unstaged run): straight to the global matrix.  row = BAM nibble, or AMP7_DEL_CODE
#define AMP7_DEL_CODE 17
AMP_HD void count_global7(const KParams& P, int* cnt, int wbase, int row, int p, unsigned& errs) {
    const unsigned w = (unsigned)(p - wbase);
    if (wbase >= 0 && w < (unsigned)P.wt) { atomic_add(&cnt[(row == AMP7_DEL_CODE ? del_row_off(P.wt) : row * P.wt) + (int)w], 1); return; }
    const int ch = row == AMP7_DEL_CODE ? 5 : row_channel(row);
    if (ch < 0) { errs |= AMP_E_BASE; return; }
    atomic_add(&P.counts[(size_t)ch * P.Lpad + p], 1);
}

// count the warp's run list [0, n_runs), 32 runs at a time (one per lane): staged aligned runs inside the tile go through
// the balanced chunk loop of the fast kernel; deletion runs and everything else are counted base by base by their lane
template <int WT>
AMP_WD void count_warp_runs7(const KParams& P, int* cnt, int wt, const WarpMem7& wm, int n_runs, int wbase, int lane, unsigned minq4) {
    const int minq = P.tp.min_quality;
    unsigned errs = 0;
    for (int base = 0; base < n_runs; base += 32) {
        int a0 = 0, n0 = 0, m = 0, w0 = 0;
        bool has = false;
        if (base + lane < n_runs) {
            const Seg sg = wm.runs[base + lane];
            const int n = sg.len & 0x3FFFFFFF;
            w0 = sg.rpos - wbase;
            const bool in_win = wbase >= 0 && w0 >= 0 && w0 + n <= wt;
            if (sg.len < 0) {                                                      // D / N run: unconditional (714-715)
                if (in_win) { for (int j = 0; j < n; ++j) atomic_add(&cnt[del_row_off(wt) + w0 + j], 1); }
                else for (int j = 0; j < n; ++j) count_global7(P, cnt, wbase, AMP7_DEL_CODE, sg.rpos + j, errs);
            } else if ((sg.len & 0x40000000) && in_win && n > 0 && n < 512 && minq >= 0 && minq <= 127) {
                a0 = (int)sg.qabs; n0 = (int)sg.nibabs; m = n; has = true;
            } else {
                const bool staged = (sg.len & 0x40000000) != 0;
                const uint8_t* qp = staged ? wm.qbuf + sg.qabs : P.b.qual + sg.qabs;
                const uint8_t* sp = staged ? wm.sbuf : P.b.seq;
                for (int j = 0; j < n; ++j) {
                    if (qp[j] < minq) continue;                                    // 718
                    const uint32_t nb = sg.nibabs + (uint32_t)j;
                    count_global7(P, cnt, wbase, (int)((sp[nb >> 1] >> ((~nb & 1u) << 2)) & 15u), sg.rpos + j, errs);   // 752-753
                }
            }
        }
        count_runs_balanced<WT>(cnt, wt, wm.qbuf, wm.sbuf, wm.par, wm.own, lane, has, a0, n0, m, w0, minq4);
    }
    if (errs) atomic_or(P.err, errs);
}

// generic path for one queued read (rows staged in slot `slot` of the warp's buffers, or read from global memory)
AMP_HD void warp_read_generic7(const KParams& P, const WarpMem7& wm, long long i, int slot, bool do_trim, bool do_pile) {
    AMP7_GT0();
    const uint32_t c0 = P.b.cig_off[i], c1 = P.b.cig_off[i + 1];
    const uint32_t qo0 = P.b.qual_off[i], qo1 = P.b.qual_off[i + 1];
    int nc = (int)(c1 - c0);
    const int l_seq = (int)(qo1 - qo0);
    const int flag = P.b.flag[i];
    int pos = P.b.pos[i];
    uint32_t so0 = 0, so1 = 0;
    if (do_pile) { so0 = P.b.seq_off[i]; so1 = P.b.seq_off[i + 1]; }
    const uint32_t qdst = AMP7_PAD + (uint32_t)slot * AMP7_GSLOT_Q + (qo0 & 15u), sdst = AMP7_PAD + (uint32_t)slot * AMP7_GSLOT_S + (so0 & 15u);
    const bool q_st = (qo0 & 15u) + (qo1 - qo0) + 16u <= AMP7_GSLOT_Q;          // row + read-ahead of the word-wise search
    const bool s_st = do_pile && (so0 & 15u) + (so1 - so0) <= AMP7_GSLOT_S;
    const uint8_t* qual = q_st ? wm.qbuf + qdst : P.b.qual + qo0;
    const uint8_t* seq = do_pile ? (s_st ? wm.sbuf + sdst : P.b.seq + so0) : nullptr;
    const uint32_t* cig = P.b.cigar + c0;
    int f = 0;
    if (do_trim) {
        uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
        // the two CIGAR work rows of trim_read live in shared memory (local-memory arrays would miss the small L1 left
        // next to the staging buffers); long CIGARs use the global scratch rows
        uint32_t *A, *B;
        if (nc + 3 <= AMP7_CROW) { A = wm.cig + (size_t)slot * 2 * AMP7_CROW; B = A + AMP7_CROW; }
        else { A = P.scratch + (size_t)c0 + 3 * (size_t)i; B = A + P.scratch_half; }
        for (int k = 0; k < nc; ++k) A[k] = cig[k];
        AMP7_GTICK(0);
        uint32_t* res;
        f = trim_read(A, B, nc, pos, flag, P.b.tlen[i], l_seq, qual, q_st, P.tp, &res);   // qdst >= AMP7_PAD >= 8
        AMP7_GTICK(1);
        if (f & AMP_F_ERROR) { nc = 0; f = AMP_F_ERROR; atomic_or(P.err, AMP_E_COORD); }
        for (int k = 0; k < nc; ++k) orow[k] = res[k];
        cig = res;
        P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = (uint8_t)f;
        AMP7_GTICK(2);
    }
    if (do_pile && !(f & AMP_F_ERROR)) {
        WarpSink7 sink; sink.P = &P; sink.wm = wm;
        sink.staged = q_st && s_st;
        sink.qabs0 = sink.staged ? qdst : qo0;
        sink.nibabs0 = sink.staged ? sdst * 2u : so0 * 2u;
        sink.seq_read = seq; sink.qual_read = qual; sink.errs = 0; sink.so0 = so0;
        int e = plan_read(cig, nc, pos, l_seq, qual, P.tp.min_quality, P.tp.L, sink);
        e |= (int)sink.errs;
        if (e) atomic_or(P.err, (unsigned)e);
        AMP7_GTICK(3);
    }
}

// G phase: the first nb (<= AMP7_GN) queued reads of the warp
template <int WT>
AMP_WD_COLD void warp_generic_phase(const KParams& P, const WarpMem7& wm, int* cnt, int wt, int wbase, int nb, int nq, int lane, bool do_trim,
                               bool do_pile, uint32_t& parity, long long* tk) {
    // stage the (scattered) rows into fixed slots, keeping each row's alignment mod 16: every lane starts the bulk copies
    // of its own read (whole 16-byte pieces, rounded up)
    {
        uint32_t qb = 0, sb = 0;
        const uint8_t *qsrc = nullptr, *ssrc = nullptr;
        uint8_t *qdst = nullptr, *sdst = nullptr;
        if (lane < nb) {
            const long long i = P.b.first + wm.queue[lane];
            const uint32_t qo0 = P.b.qual_off[i], qo1 = P.b.qual_off[i + 1];
            if ((qo0 & 15u) + (qo1 - qo0) + 16u <= AMP7_GSLOT_Q) {
                qsrc = P.b.qual + (qo0 & ~15u); qdst = wm.qbuf + AMP7_PAD + (size_t)lane * AMP7_GSLOT_Q;
                qb = ((qo0 & 15u) + (qo1 - qo0) + 15u) & ~15u;
            }
            if (do_pile) {
                const uint32_t so0 = P.b.seq_off[i], so1 = P.b.seq_off[i + 1];
                if ((so0 & 15u) + (so1 - so0) <= AMP7_GSLOT_S) {
                    ssrc = P.b.seq + (so0 & ~15u); sdst = wm.sbuf + AMP7_PAD + (size_t)lane * AMP7_GSLOT_S;
                    sb = ((so0 & 15u) + (so1 - so0) + 15u) & ~15u;
                }
            }
        }
        const uint32_t total = (uint32_t)w_add((int)(qb + sb));
        if (lane == 0) { wm.ctr[0] = 0; if (total) bulk_expect(wm.bar, total); }
        w_sync();
        if (qb) bulk_copy(qdst, qsrc, qb, wm.bar);
        if (sb) bulk_copy(sdst, ssrc, sb, wm.bar);
        w_sync();
        if (total) { bulk_wait(wm.bar, parity); parity ^= 1u; }
    }
    if (lane < nb) warp_read_generic7(P, wm, P.b.first + wm.queue[lane], lane, do_trim, do_pile);
    w_sync();
    if (do_pile) {
        int nr = wm.ctr[0]; if (nr > AMP7_RUNCAP) nr = AMP7_RUNCAP;
        count_warp_runs7<WT>(P, cnt, wt, wm, nr, wbase, lane, (unsigned)P.tp.min_quality * 0x01010101u);
    }
    // drop the processed entries (the queue holds < 64 entries: at most one move per lane and round)
    for (int base = 0; base + nb < nq; base += 32) {
        const bool mv = base + lane + nb < nq;
        const uint32_t v = mv ? wm.queue[base + lane + nb] : 0u;
        w_sync();
        if (mv) wm.queue[base + lane] = v;
        w_sync();
    }
    w_sync();
}

// an aligned run of a staged read that does not lie inside the tile: base by base, exact (rare on coordinate-sorted input)
AMP_WD_COLD void count_run_slow(const KParams& P, int* cnt, int wbase, const uint8_t* qrun, const uint8_t* sbuf, int nb0, int rpos, int m) {
    const int minq = P.tp.min_quality;
    unsigned errs = 0;
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    if (P.phase_cycles) atomicAdd((unsigned long long*)&P.phase_cycles[14], 1ULL);        // runs outside the tile
#endif
    for (int t = 0; t < m; ++t) {
        if (qrun[t] < minq) continue;                                              // 718
        const uint32_t nb = (uint32_t)(nb0 + t);
        count_global7(P, cnt, wbase, (int)((sbuf[nb >> 1] >> ((~nb & 1u) << 2)) & 15u), rpos + t, errs);   // 752-753
    }
    if (errs) atomic_or(P.err, errs);
}

// ---- the kernel ------------------------------------------------------------------------------------------------------
// P.reads_per_tile = reads per batch (<= 32), P.ntiles = batches, P.tiles_per_cta = batches per CTA (contiguous chunk).
// WT = width of the count tile as a compile-time constant (0: P.wt, used by the emulation tests).
// One CTA per SM.  Warps [0, nwarps - dwarps) work through the chunk's batches ([S]M[S] reads, phases A and B); every other
// mapped read is appended to the CTA's segment of P.glist.  The last dwarps warps (default: none) do nothing but the generic
// phase G over that list while it is being filled; the generic-capable warps work through what is left when their batches
// are done.  All of them count into the same tile.

// window base of a CTA's chunk: smallest start among its first reads (coordinate-sorted input => of the whole chunk)
AMP_WD int chunk_window_base(const KParams& P, int* ctrl, long long first_read, long long n_end, int tid, bool any) {
    if (tid == 0) ctrl[C7_TMIN] = 0x7FFFFFFF;
    c_sync();
    if (any && tid < 64) {
        const long long i = first_read + tid;
        if (i < n_end) {
            const int p0 = P.b.pos[i];
            if (p0 >= 0 && !(P.b.flag[i] & 4)) atomic_min(&ctrl[C7_TMIN], p0);
        }
    }
    c_sync();
    const int wmin = ctrl[C7_TMIN];
    return wmin != 0x7FFFFFFF ? (wmin & ~31) : -1;
}

template <bool TRIM, bool PILE, int WT>
AMP_WD void cta_trim_pileup_v9(const KParams& P, unsigned char* smem_base, int gwarps, int dwarps) {
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    const long long t_cta0 = clock64();
#endif
    const int wt = WT ? WT : P.wt;
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    const int tid = c_tid(), nthreads = c_nthreads(), block = P.direct ? (int)gridDim.x - 1 - c_block() : c_block();   // experiment: chunks in reverse order
#else
    const int tid = c_tid(), nthreads = c_nthreads(), block = c_block();
#endif
    const int lane = tid & 31, warp = tid >> 5;
    const int BR = P.reads_per_tile;
    int* cnt = (int*)smem_base;
    int* ctrl = (int*)(smem_base + tile_bytes_v7(wt));
    const FastMem wm = carve_fast(smem_base, wt, warp);
    const long long g_lo = (long long)block * P.tiles_per_cta;
    long long g_hi = g_lo + P.tiles_per_cta; if (g_hi > P.ntiles) g_hi = P.ntiles;
    const int n_batches = g_hi > g_lo ? (int)(g_hi - g_lo) : 0;
    const long long n_end = P.b.first + P.b.n;
    uint32_t* glist = P.glist + (size_t)block * P.gcap;          // overflow of the shared-memory list

    // Set-up.  The loads it depends on (start positions of the chunk's first reads for the window base, below the metadata of each
    // warp's first batch) are issued first, so that their latency overlaps the clearing of the tile and the two barriers.
    const int nwarps = nthreads >> 5, n_fast = nwarps - dwarps;     // warps [0, n_fast) take batches, the rest only the list
    int wmin0 = 0x7FFFFFFF;
    if (n_batches > 0 && tid < 64) {
        const long long i = P.b.first + g_lo * BR + tid;
        if (i < n_end) { const int p0 = P.b.pos[i]; if (p0 >= 0 && !(P.b.flag[i] & 4)) wmin0 = p0; }
    }
    if (PILE) {                                                   // the sink row is never read
        for (int i = tid; i < AMP7_SINK_ROW * wt; i += nthreads) cnt[i] = 0;
        for (int i = tid; i < wt; i += nthreads) cnt[del_row_off(wt) + i] = 0;
    }
    if (tid == 0) {
        ctrl[C7_NEXT] = n_fast;                                   // batch w is warp w's first one
        ctrl[C7_NGEN] = 0; ctrl[C7_GNEXT] = 0; ctrl[C7_FASTDONE] = 0; ctrl[C7_NEV] = 0; ctrl[C7_EVDONE] = 0; ctrl[C7_TMIN] = 0x7FFFFFFF;
    }
    for (int k = tid; k < AMP7_GLCAP; k += nthreads) ctrl[C7_GL + k] = 0;   // list entries: 0 = not written yet
    for (int k = tid; k < AMP7_EVCAP; k += nthreads) ctrl[C7_EV + 3 * k + 2] = 0;
    if (lane == 0) mbar_init(wm.bar);
    c_sync();
    if (wmin0 != 0x7FFFFFFF) atomic_min(&ctrl[C7_TMIN], wmin0);
    const int minq = P.tp.min_quality;
    // the word-wise passes need the default window and a quality threshold that fits the SIMD byte compare
    const bool fast_ok = minq >= 0 && minq <= 127 && (!TRIM || P.tp.window == 4);
    const unsigned minq4 = (unsigned)minq * 0x01010101u;
    uint32_t parity = 0;

    // Software pipeline over the warp's batches: the per-read metadata of the next batch is loaded while the current one is
    // in its window pass, its first CIGAR words (and an L2 prefetch of its rows) while the current one is being counted.
    struct Meta { uint32_t c0, c1, qo0, qo1, so0, so1; int flag, pos, tlen; uint32_t g0, g1, g2, g3, g4; };
    auto claim = [&]() -> int {
        int b = 0;
        if (lane == 0) b = atomic_add(&ctrl[C7_NEXT], 1);
        return w_shfl(b, 0);
    };
    auto read_index = [&](int b) -> long long {              // this lane's read of batch b (clamped to the batch's first read)
        const long long t0 = P.b.first + (g_lo + b) * BR;
        long long t1 = t0 + BR; if (t1 > n_end) t1 = n_end;
        return lane < (int)(t1 - t0) ? t0 + lane : t0;
    };
    auto load_meta = [&](int b, Meta& M) {
        const long long i = read_index(b);
        M.c0 = P.b.cig_off[i]; M.c1 = P.b.cig_off[i + 1];
        M.qo0 = P.b.qual_off[i]; M.qo1 = P.b.qual_off[i + 1];
        M.so0 = 0; M.so1 = 0;
        if (PILE) { M.so0 = P.b.seq_off[i]; M.so1 = P.b.seq_off[i + 1]; }
        M.flag = P.b.flag[i]; M.pos = P.b.pos[i];
        M.tlen = TRIM ? P.b.tlen[i] : 0;
    };
    auto load_cigar5 = [&](Meta& M) {
        const int nc = (int)(M.c1 - M.c0);
        M.g0 = nc > 0 ? P.b.cigar[M.c0] : 0u;
        M.g1 = nc > 1 ? P.b.cigar[M.c0 + 1] : 0u;
        M.g2 = nc > 2 ? P.b.cigar[M.c0 + 2] : 0u;
        M.g3 = nc > 3 ? P.b.cigar[M.c0 + 3] : 0u;
        M.g4 = nc > 4 ? P.b.cigar[M.c0 + 4] : 0u;
    };
    Meta M, Mn;
    M.c0 = M.c1 = M.qo0 = M.qo1 = M.so0 = M.so1 = M.g0 = M.g1 = M.g2 = M.g3 = M.g4 = 0; M.flag = M.pos = M.tlen = 0;
    Mn = M;
    int bi = warp < n_fast ? warp : n_batches;
    if (bi < n_batches) { load_meta(bi, M); load_cigar5(M); }
    c_sync();
    const int wb = ctrl[C7_TMIN] != 0x7FFFFFFF ? (ctrl[C7_TMIN] & ~31) : -1;
    const int wbase = PILE ? wb : -1;
    // the stretch of the two primer tables this chunk looks at (from its window base), for phase A
    TrimParams tps = P.tp;
    const int pbase = wb >= 0 ? wb : 0;
    if (TRIM) {
        int* ptab = ctrl + C7_PTAB;
        for (int k = tid; k < 2 * AMP7_PSLICE; k += nthreads) {
            const int p = pbase + (k < AMP7_PSLICE ? k : k - AMP7_PSLICE);
            ptab[k] = p < P.tp.L ? (k < AMP7_PSLICE ? P.tp.min_primer_start[p] : P.tp.max_primer_end[p]) : -1;
        }
        tps.min_primer_start = ptab - pbase; tps.max_primer_end = ptab + AMP7_PSLICE - pbase;
        c_sync();
    }
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    if (tid == 0 && P.phase_cycles) atomicAdd((unsigned long long*)&P.phase_cycles[11], (unsigned long long)(clock64() - t_cta0));   // set-up
#endif
    AMP7_T0(tk);
    AMP7_TICK(tk, 0);
    // One round of the generic phase: up to AMP7_GN listed reads, taken by a generic-capable warp between two of its batches
    // (wait = false: only what is there) or when its batches are done (wait = true: until the list is complete and empty).
    const bool is_gwarp = warp >= nwarps - gwarps;
    const WarpMem7 gm = carve_warp7(smem_base, wt, nwarps, gwarps, is_gwarp ? warp - (nwarps - gwarps) : 0);
    auto generic_round = [&](bool wait) -> bool {
        int at = -1, n = 0;
        if (lane == 0) {
            for (;;) {
                const bool done = ld_vol(&ctrl[C7_FASTDONE]) >= n_fast;     // read before the counters: then they are final
                const int reserved = ld_vol(&ctrl[C7_NGEN]), claimed = ld_vol(&ctrl[C7_GNEXT]);
                int avail = reserved - claimed;
                if (claimed < AMP7_GLCAP) { if (avail > AMP7_GLCAP - claimed) avail = AMP7_GLCAP - claimed; }
                else if (!done) avail = 0;
                if (avail > 0) {
                    n = avail < AMP7_GN ? avail : AMP7_GN;
                    if (atomic_cas(&ctrl[C7_GNEXT], claimed, claimed + n) == claimed) { at = claimed; break; }
                    continue;
                }
                if (done || !wait) break;
                c_yield();
            }
        }
        at = w_shfl(at, 0); n = w_shfl(n, 0);
        if (at < 0) return false;
        fence_block();
        if (lane < n) {
            const int idx = at + lane;
            uint32_t v;
            if (idx < AMP7_GLCAP) { while ((v = (uint32_t)ld_vol(&ctrl[C7_GL + idx])) == 0u) c_yield(); }   // reserved but not yet written
            else v = ld_cg_u32(&glist[idx - AMP7_GLCAP]);
            gm.queue[lane] = v - 1u;
        }
        w_sync();
        warp_generic_phase<WT>(P, gm, cnt, wt, wbase, n, n, lane, TRIM, PILE, parity, tk);
        return true;
    };
    while (bi < n_batches) {
        const long long t0 = P.b.first + (g_lo + bi) * BR;
        long long t1 = t0 + BR; if (t1 > n_end) t1 = n_end;
        const int nreads = (int)(t1 - t0);
        const bool have = lane < nreads;
        const long long i = have ? t0 + lane : t0;

        // ---- A: staging + classification (metadata already in registers) -------------------------------------------------
        const uint32_t c0 = M.c0, c1 = M.c1, qo0 = M.qo0, qo1 = M.qo1, so0 = M.so0, so1 = M.so1;
        const int flag = M.flag, tlen = M.tlen;
        int pos = M.pos;
        // staged byte ranges [lo, hi) of the batch: rows of consecutive reads are contiguous
        const uint32_t q_lo = (uint32_t)w_shfl((int)qo0, 0) & ~15u, q_end = (uint32_t)w_shfl((int)qo1, nreads - 1);
        const uint32_t q_hi = (q_end - q_lo <= (uint32_t)AMP7_QDATA) ? q_end : q_lo + (uint32_t)AMP7_QDATA;
        uint32_t s_lo = 0, s_hi = 0;
        if (PILE) {
            s_lo = (uint32_t)w_shfl((int)so0, 0) & ~15u;
            const uint32_t s_end = (uint32_t)w_shfl((int)so1, nreads - 1);
            s_hi = (s_end - s_lo <= (uint32_t)AMP7_SDATA) ? s_end : s_lo + (uint32_t)AMP7_SDATA;
        }
        // whole 16-byte pieces, rounded up: the arrays are readable up to the next 16-byte boundary (include/amplipy_b200.h)
        const uint32_t q_bulk = (q_hi - q_lo + 15u) & ~15u, s_bulk = (s_hi - s_lo + 15u) & ~15u;
        if (lane == 0 && q_bulk + s_bulk > 0) {
            bulk_expect(wm.bar, q_bulk + s_bulk);
            if (q_bulk) bulk_copy(wm.qbuf + AMP7_PAD, P.b.qual + q_lo, q_bulk, wm.bar);
            if (s_bulk) bulk_copy(wm.sbuf + AMP7_PAD, P.b.seq + s_lo, s_bulk, wm.bar);
        }

        const int nc = (int)(c1 - c0), l_seq = (int)(qo1 - qo0);
        const uint32_t* cig = P.b.cigar + c0;
        const bool skipped = have && ((flag & 4) || nc == 0);                          // AmpliPy.py:902
        Shape5 r = {0, 0, 0, 0, 0, 0, 0, 0u};
        int f = 0;
        bool fast = have && !skipped && fast_ok && qo1 <= q_hi && (!PILE || so1 <= s_hi) &&
                    classify_shape5(nc, M.g0, M.g1, M.g2, M.g3, M.g4, l_seq, r);
        if (fast && TRIM) {   // both lookups (pos and reference_end - 1) inside the cached stretch?
            const bool in_slice = pos >= pbase && pos + shape_rlen(r) <= pbase + AMP7_PSLICE;
            fast = trim_shape_primers(r, pos, flag, tlen, l_seq, in_slice ? tps : P.tp, &f);
        }
        if (fast && !TRIM && (pos < 0 || pos + shape_rlen(r) > P.tp.L)) fast = false;
        const int qrow = (int)(AMP7_PAD + (qo0 - q_lo));                               // the read's first quality byte in qbuf
        const int a0 = qrow + r.s1;                                                    // first aligned quality byte
        const int qlen = shape_qlen(r);                                                // aligned query bases (561-563)
        if (fast && (qlen < 8 || (a0 & 3) + qlen > 256)) fast = false;
        const bool rev = (flag & 16) != 0;
        // everything else goes to the CTA's list for the generic phase
        {
            const bool gen = have && !skipped && !fast;
            const unsigned gmask = w_ballot(gen);
            if (gmask) {
                int base = 0;
                if (lane == 0) base = atomic_add(&ctrl[C7_NGEN], popc32(gmask));
                base = w_shfl(base, 0);
                if (gen) {
                    const int idx = base + popc32(gmask & ((1u << lane) - 1u));
                    const uint32_t v = (uint32_t)(i - P.b.first) + 1u;                 // 0 = not written yet
                    if (idx < AMP7_GLCAP) st_vol(&ctrl[C7_GL + idx], (int)v); else st_cg_u32(&glist[idx - AMP7_GLCAP], v);
                }
            }
        }
        if (skipped && TRIM) {
            uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
            for (int k = 0; k < nc; ++k) orow[k] = cig[k];
            P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)nc; P.o.flags[i] = (uint8_t)AMP_F_SKIPPED;
        }
#if !defined(__CUDA_ARCH__)
        if (fast) ++g_v7_stats[0]; else if (have && !skipped) ++g_v7_stats[1];
#endif
        w_sync();
        AMP7_TICK(tk, 1);
        if (q_bulk + s_bulk > 0) { bulk_wait(wm.bar, parity); parity ^= 1u; }
        AMP7_TICK(tk, 2);
        const int bn = claim();                                        // next batch: its metadata loads fly during B1
        if (bn < n_batches) load_meta(bn, Mn);

        // ---- B1: lane per read: window search, quality clip + write gate + outputs; the read's runs for pass B2 -------------
        bool in1 = false, in2 = false;                                 // this lane's first / second aligned run is counted in the tile
        int qa1 = 0, nb1 = 0, w1 = 0, m1 = 0, qa2 = 0, nb2 = 0, w2 = 0, m2 = 0;
        if (fast) {
            if (TRIM) {
                const int del = window_del_blocks(wm.qbuf, a0, qlen, rev, minq);
                trim_shape_finish(r, del, rev, P.tp, &f);                             // 589-686 (pos stays on the reverse strand, F6), 910
                uint32_t* orow = P.o.cigar + (size_t)c0 + 3 * (size_t)i;
                const int no = emit_shape5(r, orow);
                P.o.pos[i] = pos; P.o.ncig[i] = (uint16_t)no; P.o.flags[i] = (uint8_t)f;
            }
            if (PILE) {
                // final shape [S] M [I|D] [M] [S] at pos: walk it as update_base_counts walks the aligned pairs
                const int nrow = (int)(2u * (AMP7_PAD + so0 - s_lo));                 // nibble index of the read's first base in sbuf
                unsigned errs = 0;
                int q = r.s1, rp = pos;
                m1 = r.m; qa1 = qrow + q; nb1 = nrow + q; w1 = rp - wbase;
                q += r.m; rp += r.m;
                if (r.k > 0) {
                    if (shape_xop(r) == OP_D) {                                       // 714-715
                        for (int j = 0; j < r.k; ++j) count_global7(P, cnt, wbase, AMP7_DEL_CODE, rp + j, errs);
                        rp += r.k;
                    } else {
                        auto emit = [&](int ipos, int b, int n) { ins_defer(P, ctrl, so0, ipos, b, n); };
                        shape_ins_events(r, pos, l_seq, wm.qbuf + qrow, minq, emit);  // 730-748
                        q += r.k;
                    }
                }
                m2 = r.m2; qa2 = qrow + q; nb2 = nrow + q; w2 = rp - wbase;
                if (m1 <= 0) { m1 = m2; qa1 = qa2; nb1 = nb2; w1 = w2; m2 = 0; }
                in1 = m1 > 0 && wbase >= 0 && w1 >= 0 && w1 + m1 <= wt;
                in2 = m2 > 0 && wbase >= 0 && w2 >= 0 && w2 + m2 <= wt;
                // outside the tile: base by base into the global matrix (exact, rare on sorted input)
                if (m1 > 0 && !in1) count_run_slow(P, cnt, wbase, wm.qbuf + qa1, wm.sbuf, nb1, w1 + wbase, m1);
                if (m2 > 0 && !in2) count_run_slow(P, cnt, wbase, wm.qbuf + qa2, wm.sbuf, nb2, w2 + wbase, m2);
                if (errs) atomic_or(P.err, errs);
            }
        }
        AMP7_TICK(tk, 3);
        if (bn < n_batches) {                                          // stage 2 of the next batch: CIGAR words, rows towards L2
            load_cigar5(Mn);
            const long long tn0 = P.b.first + (g_lo + bn) * BR;
            long long tn1 = tn0 + BR; if (tn1 > n_end) tn1 = n_end;
            const uint32_t pq_lo = (uint32_t)w_shfl((int)Mn.qo0, 0) & ~15u, pq_hi = (uint32_t)w_shfl((int)Mn.qo1, (int)(tn1 - tn0) - 1);
            const uint32_t ps_lo = (uint32_t)w_shfl((int)Mn.so0, 0) & ~15u, ps_hi = (uint32_t)w_shfl((int)Mn.so1, (int)(tn1 - tn0) - 1);
            if (lane == 0) {
                uint32_t nq = (pq_hi - pq_lo) & ~15u; if (nq > (uint32_t)AMP7_QDATA) nq = AMP7_QDATA;
                if (nq) bulk_prefetch_l2(P.b.qual + pq_lo, nq);
                uint32_t ns = (ps_hi - ps_lo) & ~15u; if (ns > (uint32_t)AMP7_SDATA) ns = AMP7_SDATA;
                if (PILE && ns) bulk_prefetch_l2(P.b.seq + ps_lo, ns);
            }
        }
        // ---- B2: pileup of the batch's aligned runs, chunks dealt out evenly over the lanes ----------------------------------
        if (PILE) {   // (one call site: the loop body is the kernel's hottest code and should exist once)
            const int npass = w_ballot(in2) ? 2 : 1;
            for (int pass = 0; pass < npass; ++pass) {
                count_runs_balanced<WT>(cnt, wt, wm.qbuf, wm.sbuf, wm.par, wm.own, lane, pass ? in2 : in1, pass ? qa2 : qa1, pass ? nb2 : nb1,
                                        pass ? m2 : m1, pass ? w2 : w1, minq4);
            }
        }
        w_sync();   // every lane is done with the staged rows before the buffers are reused
        AMP7_TICK(tk, 4);
        M = Mn; bi = bn;
    }
    AMP7_TICK(tk, 5);
    if (warp < n_fast) { fence_block(); if (lane == 0) atomic_add(&ctrl[C7_FASTDONE], 1); }   // this warp appends no more
    // ---- G: whatever is left of the list (entries in shared memory are taken while the list is still being filled, the
    // overflow in global memory once every batch warp is done), then the parked insertion alleles
    if (is_gwarp) while (generic_round(true)) {}
    if (PILE) ins_drain(P, ctrl, lane);
    AMP7_TICK(tk, 6);
    AMP7_TDUMP(tk, 0);
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    const long long t_bar0 = clock64();
#endif
    c_sync();
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    const long long t_bar1 = clock64();
    if (lane == 0 && P.phase_cycles) atomicAdd((unsigned long long*)&P.phase_cycles[12], (unsigned long long)(t_bar1 - t_bar0));     // wait at the last barrier, per warp
#endif
    if (PILE) ins_drain(P, ctrl, lane);                            // alleles parked by the last warps to finish
    if (PILE && wbase >= 0) flush_tile7(P, cnt, wbase, tid, nthreads);
#if defined(__CUDA_ARCH__) && defined(AMP7_TIMING)
    if (tid == 0 && P.phase_cycles) {   // whole-CTA cycles: sum / min / max over CTAs
        const long long tot = clock64() - t_cta0;
        atomicAdd((unsigned long long*)&P.phase_cycles[13], (unsigned long long)(clock64() - t_bar1));                               // drain + flush (thread 0's view)
        atomicAdd((unsigned long long*)&P.phase_cycles[8], (unsigned long long)tot);
        atomicMin((long long*)&P.phase_cycles[9], tot);
        atomicMax((long long*)&P.phase_cycles[10], tot);
        if (block < 160) { P.phase_cycles[16 + block] = tot; P.phase_cycles[176 + block] = ctrl[C7_NGEN]; }
    }
#endif
}

}  // namespace amp
