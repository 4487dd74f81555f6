// amp_ivar.cuh -- iVar-format outputs (DESIGN.md 3.7): a strand / quality pass over the reads the pileup counted, and the
// calling that turns its sums into mean qualities, Fisher p-values and an IUPAC-ambiguity consensus.  Written as
// __host__ __device__ code so that tests/emu runs this very source on the CPU.
//
//   cta_qstats     one CTA per AMP_QS_READS coordinate-sorted reads, one thread per read: plan_read (amp_core.cuh) walks the
//                  CIGAR the pileup walked (the trimmed row when trimming ran) and a sink adds, for every event the count matrix
//                  received, 1 to rev when the read is on the reverse strand and the base's phred quality to qsum (A C G T N; the
//                  '-' row carries no quality, 714-715).  A privatised tile over the CTA's reference window takes what falls in
//                  it and is flushed with global atomics; whatever falls outside goes straight to global memory.
//                  cta_qstats<true> also adds every anchored deletion event to the deletion-allele table (amp_dels.cuh).
//   ivar_position  one thread per (sample, position), after amp_call on its outputs.
//   ivar_del       one thread per deletion allele, after amp_call on its depths.
#pragma once
#include <math.h>

#include "amp_kernels.cuh"
#include "amp_dels.cuh"

namespace amp {

#define AMP_QS_READS 256     // reads per CTA of the strand / quality pass (one per thread)
#define AMP_QS_WT 768        // reference positions of its privatised tile (2 x 6 x 768 ints = 36 KB)

struct QStatsParams {
    BatchPtrs b;
    TrimOut o; int trimmed;                    // trimmed: the rows of `o` are the ones the pileup walked
    int L, Lpad, minq, gpos_base;
    int* rev; unsigned long long* qsum;         // this sample's [6][Lpad]
    InsTable tab;                               // looked up only: every allele was added by the fused kernel
    int* ins_rev; unsigned long long* ins_qsum; // per slot
    unsigned char* ins_head;                    // per slot: 1 = an event of this allele is the key of 735-736
    unsigned int* err;
    DelTable dels;                              // cta_qstats<true> only: the anchored deletion alleles
};

// DELS: anchored deletion events also go to P->dels (a separate instance, so the pass without the table is unchanged)
template <bool DELS = false>
struct QStatsSink {
    const QStatsParams* P; int* trev; int* tq; int wbase;
    const uint8_t* seq; const uint8_t* qual; bool rev; unsigned int errs;
    // one event at (ch, p) of quality q (0 for '-')
    AMP_HD void add(int ch, int p, int q) {
        const unsigned w = (unsigned)(p - wbase);
        if (wbase >= 0 && w < (unsigned)AMP_QS_WT) {
            if (rev) atomic_add(&trev[ch * AMP_QS_WT + (int)w], 1);
            if (q) atomic_add(&tq[ch * AMP_QS_WT + (int)w], q);
        } else {
            const size_t o = (size_t)ch * P->Lpad + p;
            if (rev) atomic_add(&P->rev[o], 1);
            if (q) atomic_add64(&P->qsum[o], (unsigned long long)q);
        }
    }
    AMP_HD void match(int rpos, int q, int n) {
        for (int j = 0; j < n; ++j) {
            const int qv = qual[q + j];
            if (qv < P->minq) continue;                                           // 718
            const int ch = nib_channel(nib_at(seq, (uint32_t)(q + j)));
            if (ch >= 0) add(ch, rpos + j, qv);                                   // 752-753 (a KeyError is the pileup's to raise)
        }
    }
    AMP_HD void del(int rpos, int n, int qa) {
        if (rev) for (int j = 0; j < n; ++j) add(5, rpos + j, 0);                                      // 714-715
        if (DELS && qa >= 0) {                                                    // an anchored deletion (DESIGN.md 3.7)
            const int aq = qual[qa];
            if (aq >= P->minq) del_table_add(P->dels, P->gpos_base + rpos - 1, n, 1u, rev ? 1u : 0u, (unsigned long long)aq);
        }
    }
    AMP_HD void ins(int pos, int b, int n, int q0) {
        const int eq = qual[q0];                                                  // the first inserted base past 718 / 722
        if (n == 1) {
            const int ch = nib_channel(nib_at(seq, (uint32_t)b));
            if (ch >= 0) { add(ch, pos, eq); return; }                            // the base's own counter (745-746)
        }
        TileSink::Text t; t.seq = seq; t.b = b;
        const int slot = ins_table_find(P->tab, P->gpos_base + pos, n, t);
        if (slot < 0) { errs |= AMP_E_QSTATS_MISS; return; }
        if (rev) atomic_add(&P->ins_rev[slot], 1);
        atomic_add64(&P->ins_qsum[slot], (unsigned long long)eq);
        if (b == q0) P->ins_head[slot] = 1;
    }
};

// the CIGAR row read i was piled up with; false: the pileup skipped it (902, or a trim result SKIPPED / ERROR)
AMP_HD bool qstats_row(const QStatsParams& P, long long i, const uint32_t*& cig, int& nc, int& pos) {
    const uint32_t c0 = P.b.cig_off[i];
    if (P.trimmed) {
        if (P.o.flags[i] & (AMP_F_SKIPPED | AMP_F_ERROR)) return false;
        cig = P.o.cigar + (size_t)c0 + 3 * (size_t)i; nc = P.o.ncig[i]; pos = P.o.pos[i];
    } else {
        cig = P.b.cigar + c0; nc = (int)(P.b.cig_off[i + 1] - c0); pos = P.b.pos[i];
    }
    return !((P.b.flag[i] & 4) || nc == 0);
}

// trev / tq: the tile, 6 x AMP_QS_WT ints each; lo: one shared int
template <bool DELS = false>
AMP_HD void cta_qstats(const QStatsParams& P, int* trev, int* tq, int* lo, int block, int nthreads) {
    const long long r0 = P.b.first + (long long)block * AMP_QS_READS;
    long long r1 = r0 + AMP_QS_READS; if (r1 > P.b.first + P.b.n) r1 = P.b.first + P.b.n;
    AMP_FOR_THREADS(tid, nthreads) {
        for (int k = tid; k < AMP_NCH * AMP_QS_WT; k += nthreads) { trev[k] = 0; tq[k] = 0; }
        if (tid == 0) *lo = 0x7FFFFFFF;
    }
    AMP_SYNC();
    AMP_FOR_THREADS(tid, nthreads) {                       // the window starts at the CTA's first read (reads are sorted)
        for (long long i = r0 + tid; i < r1; i += nthreads) {
            const uint32_t* cig; int nc, pos;
            if (qstats_row(P, i, cig, nc, pos) && pos >= 0) atomic_min(lo, pos);
        }
    }
    AMP_SYNC();
    const int wbase = *lo == 0x7FFFFFFF ? -1 : (*lo & ~31);
    AMP_FOR_THREADS(tid, nthreads) {
        unsigned int errs = 0;
        for (long long i = r0 + tid; i < r1; i += nthreads) {
            const uint32_t* cig; int nc, pos;
            if (!qstats_row(P, i, cig, nc, pos)) continue;
            QStatsSink<DELS> s;
            s.P = &P; s.trev = trev; s.tq = tq; s.wbase = wbase;
            s.seq = P.b.seq + P.b.seq_off[i]; s.qual = P.b.qual + P.b.qual_off[i];
            s.rev = (P.b.flag[i] & 16) != 0; s.errs = 0;
            plan_read(cig, nc, pos, (int)(P.b.qual_off[i + 1] - P.b.qual_off[i]), s.qual, P.minq, P.L, s);   // its errors are the pileup's
            errs |= s.errs;
        }
        if (errs) atomic_or(P.err, errs);
    }
    AMP_SYNC();
    if (wbase < 0) return;
    AMP_FOR_THREADS(tid, nthreads) {
        for (int k = tid; k < AMP_NCH * AMP_QS_WT; k += nthreads) {
            const int ch = k / AMP_QS_WT, p = wbase + k % AMP_QS_WT;
            const size_t o = (size_t)ch * P.Lpad + p;
            if (trev[k]) atomic_add(&P.rev[o], trev[k]);
            if (tq[k]) atomic_add64(&P.qsum[o], (unsigned long long)(unsigned int)tq[k]);
        }
    }
}

// ---- calling ---------------------------------------------------------------------------------------------------------------
// 10 ** (-q / 10) as python evaluates it, q = 0 .. 255: the expected error count floor(D * 10^(-mq/10)) is the same here, on
// the device and in a python reference
#define AMP_POW10_INIT \
    0x1.0000000000000p+0, 0x1.96b230bcdc434p-1, 0x1.430cd74f6d478p-1, 0x1.009b9cf334252p-1, 0x1.97a967f7524b2p-2, 0x1.43d136248490fp-2, \
    0x1.0137987dd704cp-2, 0x1.98a13577c93c0p-3, 0x1.44960c576b375p-3, 0x1.01d3f2d9684d0p-3, 0x1.999999999999ap-4, 0x1.455b5a30b035cp-4, \
    0x1.0270ac3f8a9fap-4, 0x1.9a9294b8536e9p-5, 0x1.46211ff90ea2ap-5, 0x1.030dc4ea03a72p-5, 0x1.9b8c272fbe6dep-6, 0x1.46e75df96dc9ap-6, \
    0x1.03ab3d12bc2c4p-6, 0x1.9c86515bda14ep-7, 0x1.47ae147ae147bp-7, 0x1.044914f3c02b0p-7, 0x1.9d811398ddcc0p-8, 0x1.487543c6a9257p-8, \
    0x1.04e74cc73ee88p-8, 0x1.9e7c6e43390b7p-9, 0x1.493cec2631f18p-9, 0x1.0585e4c78b079p-9, 0x1.9f7861b7937a3p-10, 0x1.4a050de314dd8p-10, \
    0x1.0624dd2f1a9fcp-10, 0x1.a074ee52cd119p-11, 0x1.4acda94717d66p-11, 0x1.06c4363887513p-11, 0x1.a1721471fe40dp-12, 0x1.4b96be9c2da2cp-12, \
    0x1.0763f01e8e5adp-12, 0x1.a26fd472780c1p-13, 0x1.4c604e2c75fb6p-13, 0x1.08040b1c10b13p-13, 0x1.a36e2eb1c432dp-14, 0x1.4d2a58423da81p-14, \
    0x1.08a4876c1311ep-14, 0x1.a46d238da54ebp-15, 0x1.4df4dd27fe99ep-15, 0x1.09456549be1bdp-15, 0x1.a56cb36416f83p-16, 0x1.4ebfdd286009ap-16, \
    0x1.09e6a4f05e62bp-16, 0x1.a66cde934de7dp-17, 0x1.4f8b588e368f1p-17, 0x1.0a88469b64867p-17, 0x1.a76da579b81cap-18, 0x1.50574fa4843efp-18, \
    0x1.0b2a4a866547ep-18, 0x1.a86f0875fcf94p-19, 0x1.5123c2b678c69p-19, 0x1.0bccb0ed19a15p-19, 0x1.a97107e6fd6abp-20, 0x1.51f0b20f71864p-20, \
    0x1.0c6f7a0b5ed8dp-20, 0x1.aa73a42bd40a5p-21, 0x1.52be1dfaf9b08p-21, 0x1.0d12a61d3698cp-21, 0x1.ab76dda3d53fdp-22, 0x1.538c06c4ca610p-22, \
    0x1.0db6355ec7054p-22, 0x1.ac7ab4ae8f688p-23, 0x1.545a6cb8cabbcp-23, 0x1.0e5a280c5ad1dp-23, 0x1.ad7f29abcaf48p-24, 0x1.5529502310084p-24, \
    0x1.0efe7e62615a0p-24, 0x1.ae843cfb8a8e0p-25, 0x1.55f8b14fddccap-25, 0x1.0fa3389d6eb40p-25, 0x1.af89eefe0b3b9p-26, 0x1.56c8908ba5ed3p-26, \
    0x1.104856fa3bc97p-26, 0x1.b0904013c482ep-27, 0x1.5798ee2308c3ap-27, 0x1.10edd9b5a66d0p-27, 0x1.b197309d68910p-28, 0x1.5869ca62d53dap-28, \
    0x1.1193c10cb1708p-28, 0x1.b29ec0fbe4534p-29, 0x1.593b259808fc7p-29, 0x1.123a0d3c84be6p-29, 0x1.b3a6f1905fa7bp-30, 0x1.5a0d000fd068cp-30, \
    0x1.12e0be826d695p-30, 0x1.b4afc2bc3d7b3p-31, 0x1.5adf5a1786da6p-31, 0x1.1387d51bddcaep-31, 0x1.b5b934e11be74p-32, 0x1.5bb233fcb6a90p-32, \
    0x1.142f51466d96cp-32, 0x1.b6c34860d463dp-33, 0x1.5c858e0d1952fp-33, 0x1.14d7333fd9ed6p-33, 0x1.b7cdfd9d7bdbbp-34, 0x1.5d5968969795cp-34, \
    0x1.157f7b46057b8p-34, 0x1.b8d954f962de4p-35, 0x1.5e2dc3e74985dp-35, 0x1.16282996f8873p-35, 0x1.b9e54ed715be1p-36, 0x1.5f02a04d76b64p-36, \
    0x1.16d13e70e10f2p-36, 0x1.baf1eb995caf0p-37, 0x1.5fd7fe1796495p-37, 0x1.177aba1212de3p-37, 0x1.bbff2ba33bf8dp-38, 0x1.60addd944f183p-38, \
    0x1.18249cb9079e4p-38, 0x1.bd0d0f57f40b8p-39, 0x1.61843f1277cb4p-39, 0x1.18cee6a45ef83p-39, 0x1.be1b971b01b1ep-40, 0x1.625b22e116f26p-40, \
    0x1.19799812dea11p-40, 0x1.bf2ac3501e305p-41, 0x1.6332894f632d7p-41, 0x1.1a24b1437279cp-41, 0x1.c03a945b3f639p-42, 0x1.640a72acc33c6p-42, \
    0x1.1ad032752ca29p-42, 0x1.c14b0aa097f38p-43, 0x1.64e2df48ce27ep-43, 0x1.1b7c1be7458ecp-43, 0x1.c25c268497682p-44, 0x1.65bbcf734b59ep-44, \
    0x1.1c286dd91c246p-44, 0x1.c36de86bea5c6p-45, 0x1.6695437c32b61p-45, 0x1.1cd5288a35c9fp-45, 0x1.c48050bb7a9dcp-46, 0x1.676f3bb3acc2dp-46, \
    0x1.1d824c3a3e865p-46, 0x1.c5935fd86f4acp-47, 0x1.6849b86a12b9bp-47, 0x1.1e2fd9290914bp-47, 0x1.c6a716282d070p-48, 0x1.6924b9efeeb05p-48, \
    0x1.1eddcf968ef81p-48, 0x1.c7bb7410560fep-49, 0x1.6a004095fbb16p-49, 0x1.1f8c2fc2f09bep-49, 0x1.c8d079f6ca708p-50, 0x1.6adc4cad25d57p-50, \
    0x1.203af9ee75616p-50, 0x1.c9e62841a8211p-51, 0x1.6bb8de868a6c0p-51, 0x1.20ea2e598bc04p-51, 0x1.cafc7f574b268p-52, 0x1.6c95f673780cbp-52, \
    0x1.2199cd44c95abp-52, 0x1.cc137f9e4dc63p-53, 0x1.6d7394c56ec06p-53, 0x1.2249d6f0eb112p-53, 0x1.cd2b297d889bcp-54, 0x1.6e51b9ce2018dp-54, \
    0x1.22fa4b9ed5233p-54, 0x1.ce437d5c12cd3p-55, 0x1.6f3065df6f53ap-55, 0x1.23ab2b8f933d6p-55, 0x1.cf5c7ba14228ap-56, 0x1.700f994b716b5p-56, \
    0x1.245c77045899fp-56, 0x1.d07624b4ab50bp-57, 0x1.70ef54646d497p-57, 0x1.250e2e3e8013ep-57, 0x1.d19078fe21d1fp-58, 0x1.71cf977cdbd76p-58, \
    0x1.25c0517f8c42ep-58, 0x1.d2ab78e5b8623p-59, 0x1.72b062e768208p-59, 0x1.2672e10927891p-59, 0x1.d3c724d3c0f64p-60, 0x1.7391b6f6ef73cp-60, \
    0x1.2725dd1d243acp-60, 0x1.d4e37d30ccec9p-61, 0x1.747393fe8174cp-61, 0x1.27d945fd7cac5p-61, 0x1.d6008265ad37dp-62, 0x1.7555fa51604e8p-62, \
    0x1.288d1bec534d3p-62, 0x1.d71e34db7274fp-63, 0x1.7638ea4300c50p-63, 0x1.29415f2bf2c30p-63, 0x1.d83c94fb6d2acp-64, 0x1.771c64270a56ep-64, \
    0x1.29f60ffecdf70p-64, 0x1.d95ba32f2de08p-65, 0x1.78006851575fep-65, 0x1.2aab2ea7803edp-65, 0x1.da7b5fe085486p-66, 0x1.78e4f715f52a5p-66, \
    0x1.2b60bb68cd6a6p-66, 0x1.db9bcb79846b3p-67, 0x1.79ca10c924223p-67, 0x1.2c16b685a1df1p-67, 0x1.dcbce6647cbe6p-68, 0x1.7aafb5bf57e6cp-68, \
    0x1.2ccd204112b32p-68, 0x1.dddeb10c00648p-69, 0x1.7b95e64d376d1p-69, 0x1.2d83f8de5dbb7p-69, 0x1.df012bdae243dp-70, 0x1.7c7ca2c79d229p-70, \
    0x1.2e3b40a0e9b4fp-70, 0x1.e024573c3631cp-71, 0x1.7d63eb8396febp-71, 0x1.2ef2f7cc46524p-71, 0x1.e148339b511e9p-72, 0x1.7e4bc0d666b6dp-72, \
    0x1.2fab1ea42c574p-72, 0x1.e26cc163c92bfp-73, 0x1.7f34231581cfep-73, 0x1.3063b56c7db54p-73, 0x1.e392010175ee6p-74, 0x1.801d129691c16p-74, \
    0x1.311cbc6945989p-74, 0x1.e4b7f2e070839p-75, 0x1.81068faf74187p-75, 0x1.31d633deb8924p-75, 0x1.e5de976d13bedp-76, 0x1.81f09ab63a899p-76, \
    0x1.32901c1134a65p-76, 0x1.e705ef13fc553p-77, 0x1.82db34012b251p-77, 0x1.334a754541678p-77, 0x1.e82dfa4208f42p-78, 0x1.83c65be6c0694p-78, \
    0x1.34053fbf90139p-78, 0x1.e956b9645a83ap-79, 0x1.84b212bda9657p-79, 0x1.34c07bc4fba14p-79, 0x1.ea802ce8543d4p-80, 0x1.859e58dcc9ddcp-80, \
    0x1.357c299a88ea7p-80, 0x1.ebaa553b9bd8dp-81, 0x1.868b2e9b3a5cep-81, 0x1.3638498566baap-81, 0x1.ecd532cc19b8ep-82, 0x1.8778945048695p-82, \
    0x1.36f4dbcaedeacp-82, 0x1.ee00c607f9020p-83, 0x1.88668a5376977p-83, 0x1.37b1e0b0a17e3p-83, 0x1.ef2d0f5da7dd9p-84, 0x1.895510fc7cad7p-84, \
    0x1.386f587c2eb0bp-84, 0x1.f05a0f3bd790fp-85, 0x1.8a4428a347c72p-85, 0x1.392d43736d210p-85
#ifdef __CUDACC__
__device__ __constant__ double kPow10Dev[256] = {AMP_POW10_INIT};
#endif
static const double kPow10Host[256] = {AMP_POW10_INIT};
AMP_HD double pow10_neg_tenth(int q) {
#ifdef __CUDA_ARCH__
    return kPow10Dev[q & 255];
#else
    return kPow10Host[q & 255];
#endif
}

// P(X <= e) for X hypergeometric with the margins of [[e, D - e], [a, D - a]], e = floor(D * 10^(-mq/10)): the left tail of
// Fisher's exact test (scipy.stats.fisher_exact(table, alternative="less")).  The pmf is evaluated once with lgamma and then
// stepped outward from e with its term ratios until the terms no longer change the sum; past the mode, 1 - the right tail.
AMP_HD double fisher_less(long long D, long long a, int mq) {
    const long long e = (long long)floor((double)D * pow10_neg_tenth(mq));
    const long long K = e + a, n = D, M = 2 * D;                  // first column, first row, table total
    const long long lo = K - D > 0 ? K - D : 0, hi = K < D ? K : D;
    if (e >= hi) return 1.0;
    const double Kd = (double)K, nd = (double)n, Md = (double)M, rest = (double)(M - K - n);   // rest = D - e - a
    const double lnorm = lgamma(Md + 1.0) - lgamma(nd + 1.0) - lgamma(Md - nd + 1.0);
    auto logpmf = [&](double x) {
        return lgamma(Kd + 1.0) - lgamma(x + 1.0) - lgamma(Kd - x + 1.0) + lgamma(Md - Kd + 1.0) - lgamma(nd - x + 1.0) -
               lgamma(rest + x + 1.0) - lnorm;
    };
    const long long mode = (long long)floor((nd + 1.0) * (Kd + 1.0) / (Md + 2.0));
    double t = 1.0, s = 1.0;
    if (e <= mode) {
        for (long long x = e; x > lo; --x) {                                          // pmf(x - 1) / pmf(x)
            const double xd = (double)x;
            t *= xd * (rest + xd) / ((Kd - xd + 1.0) * (nd - xd + 1.0));
            s += t;
            if (t < s * 1e-17) break;
        }
        const double p = exp(logpmf((double)e)) * s;
        return p < 1.0 ? p : 1.0;
    }
    for (long long x = e + 1; x < hi; ++x) {                                          // pmf(x + 1) / pmf(x)
        const double xd = (double)x;
        t *= (Kd - xd) * (nd - xd) / ((xd + 1.0) * (rest + xd + 1.0));
        s += t;
        if (t < s * 1e-17) break;
    }
    const double p = 1.0 - exp(logpmf((double)(e + 1))) * s;
    return p > 0.0 ? p : 0.0;
}

struct IvarParams {
    int L, Lpad, n_samples;
    const int* counts; const unsigned long long* qsum;            // [n_samples][6][Lpad]
    const InsSlot* slots; const int* slot_entry; const unsigned char* arena; const int* heads;
    const unsigned long long* ins_qsum;                           // per slot
    const unsigned char* ref_seq; long long ref_stride;
    // amp_call's outputs
    const int* depth; const int* top_id; const int* top_count; const double* fixed_freq; const int* fixed_rank;
    const double* ins_freq; const int* ins_rank;
    int min_depth; double min_freq; double iupac_threshold;
    // outputs
    unsigned char* iupac;              // [S*L] IUPAC code, 0 = the reference's own consensus symbol
    int* fixed_mq; double* fixed_pval; // [S*L*6]; pval NaN = no TSV row
    int* ins_mq; double* ins_pval;     // [n_alleles], dense index k
};

AMP_HD Sym ivar_slot_sym(const IvarParams& P, int slot) {
    const unsigned char* rec = P.arena + (P.slots[slot].key & 0xFFFFFFFFFFULL) * 8;
    Sym s; s.p = rec + 8; s.len = (int)((const unsigned int*)rec)[1]; return s;
}

// bases A C G T as bits 0..3 -> IUPAC code
#define AMP_IUPAC_CODES "\0ACMGRSVTWYHKDBN"

AMP_HD void ivar_position(const IvarParams& P, long long gp) {
    const int sample = (int)(gp / P.L), p = (int)(gp - (long long)sample * P.L);
    const int* cnt = P.counts + (size_t)sample * AMP_NCH * P.Lpad;
    const unsigned long long* qs = P.qsum + (size_t)sample * AMP_NCH * P.Lpad;
    const int head = P.heads[(size_t)sample * P.Lpad + p];
    const long long D = P.depth[gp];
    const unsigned char refsym = P.ref_seq[(size_t)sample * (size_t)P.ref_stride + p];
    const bool rows = D > 0 && D >= P.min_depth;
    const double nan = (double)NAN;
    unsigned long long qb = 0; long long nb = 0;
    for (int ch = 0; ch < AMP_NCH - 1; ++ch) { qb += qs[(size_t)ch * P.Lpad + p]; nb += cnt[(size_t)ch * P.Lpad + p]; }
    for (int ch = 0; ch < AMP_NCH; ++ch) {
        const long long c = cnt[(size_t)ch * P.Lpad + p];
        const int mq = ch < AMP_NCH - 1 ? (c ? (int)(qs[(size_t)ch * P.Lpad + p] / (unsigned long long)c) : 0)
                                        : (nb ? (int)(qb / (unsigned long long)nb) : 0);   // '-': the position's mean base quality
        P.fixed_mq[gp * AMP_NCH + ch] = mq;
        const bool row = rows && c && (unsigned char)"ACGTN-"[ch] != refsym && P.fixed_freq[gp * AMP_NCH + ch] >= P.min_freq;
        P.fixed_pval[gp * AMP_NCH + ch] = row ? fisher_less(D, c, mq) : nan;
    }
    for (int s = head; s >= 0; s = P.slots[s].next) {
        const long long c = P.slots[s].count;
        const int k = P.slot_entry[s];
        const int mq = c ? (int)(P.ins_qsum[s] / (unsigned long long)c) : 0;
        P.ins_mq[k] = mq;
        const Sym me = ivar_slot_sym(P, s);
        const bool row = rows && c && me.len > 0 && !(me.len == 1 && me.p[0] == refsym) && P.ins_freq[k] >= P.min_freq;
        P.ins_pval[k] = row ? fisher_less(D, c, mq) : nan;
    }
    // IUPAC: the shortest prefix of the sorted allele list whose frequencies reach the threshold
    unsigned char code = 0;
    const int tc = P.top_count[gp];
    if (P.top_id[gp] >= 0 && tc >= P.min_depth && (double)tc / (double)D >= P.min_freq) {            // 928
        double sum = 0.0; int n = 0; unsigned mask = 0; bool has_n = false;
        for (int r = 0;; ++r) {
            int id = -1; double f = 0.0;
            for (int ch = 0; ch < AMP_NCH && id < 0; ++ch)
                if (P.fixed_rank[gp * AMP_NCH + ch] == r) { id = ch; f = P.fixed_freq[gp * AMP_NCH + ch]; }
            for (int s = head; s >= 0 && id < 0; s = P.slots[s].next) {
                const int k = P.slot_entry[s];
                if (P.slots[s].count && P.ins_rank[k] == r) { id = AMP_NCH; f = P.ins_freq[k]; }
            }
            if (id < 0) break;
            sum += f; ++n;
            if (id < 4) mask |= 1u << id;
            else if (id == 4) has_n = true;
            if (sum >= P.iupac_threshold) break;
        }
        if (n > 1) code = has_n ? (unsigned char)'N' : (unsigned char)AMP_IUPAC_CODES[mask];
    }
    P.iupac[gp] = code;
}

struct IvarDelParams {
    int L, Lpad;
    DelTable dels; unsigned long long n;           // the first n listed alleles
    const int* depth;                              // amp_call's, [n_samples * L]
    int min_depth; double min_freq;
    int* mq; double* pval;                         // [n] in list order; pval NaN = no TSV row
};

// Deletion allele k: mq = floor(qsum / count) and, when it gets a TSV row (D > 0, D >= min_depth, count / D >= min_freq, D the
// depth at the anchor), PVAL = fisher_less(D, count, mq).
AMP_HD void ivar_del(const IvarDelParams& P, unsigned long long k) {
    const DelSlot& s = P.dels.slots[P.dels.entries[k]];
    int sample, a, len;
    del_key_split(s.key, P.Lpad, sample, a, len);
    const long long c = (long long)(s.cr & 0xFFFFFFFFULL);
    const long long D = P.depth[(size_t)sample * P.L + a];
    const int mq = c ? (int)(s.qsum / (unsigned long long)c) : 0;
    P.mq[k] = mq;
    const bool row = D > 0 && D >= P.min_depth && c && (double)c / (double)D >= P.min_freq;
    P.pval[k] = row ? fisher_less(D, c, mq) : (double)NAN;
}

}  // namespace amp
