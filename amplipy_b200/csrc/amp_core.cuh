// amp_core.cuh -- per-read device logic of the trim -> pileup path (sm_100a), written as
// __host__ __device__ code so that tests/emu can execute the very same source on the CPU.
//
// Reference behaviour being reproduced (file:line in /root/reference/AmpliPy.py):
//   get_pos_on_ref 363-386, get_pos_on_query 389-412, fix_cigar 415-423, trim_read 426-687,
//   update_base_counts 690-753.  pysam-derived quantities (reference_end, query_alignment_start/
//   end, get_aligned_pairs) follow pysam 0.17 / htslib semantics (SURVEY.md section 8c).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define AMP_HD __host__ __device__ __forceinline__
#define AMP_HD_NOINLINE __host__ __device__ __noinline__
#else
#define AMP_HD inline
#define AMP_HD_NOINLINE inline
#endif

// ---- out_flags bits (include/amplipy_b200.h) -------------------------------------------------
#define AMP_F_TRIM_START 1
#define AMP_F_TRIM_END 2
#define AMP_F_TRIM_QUAL 4
#define AMP_F_KEEP 8
#define AMP_F_SKIPPED 16
#define AMP_F_ERROR 32

// ---- device error word bits -------------------------------------------------------------------
#define AMP_E_COORD 1        // read outside the genome (IndexError in the reference)
#define AMP_E_BASE 2         // aligned base not in ACGTN (KeyError in the reference)
#define AMP_E_INS_END 4      // insertion run reaches the end of the pair list (IndexError, 734)
#define AMP_E_CIGAR 8        // query-consuming ops exceed l_seq / unsupported op
#define AMP_E_TABLE_FULL 16  // insertion hash table full
#define AMP_E_ARENA_FULL 32  // insertion string arena full
#define AMP_E_QSTATS_MISS 64 // strand / quality pass: an insertion allele the pileup did not add (amp_ivar.cuh)

#define AMP_NCH 6            // channels A C G T N '-'

#ifndef __CUDACC__
struct uint4 { unsigned int x, y, z, w; };   // host emulation build only
#endif

#define AMP_PRAGMA_X(x) _Pragma(#x)
#define AMP_UNROLL_N(n) AMP_PRAGMA_X(unroll n)
#if defined(__CUDACC__)
#define AMP_UNROLL AMP_PRAGMA_X(unroll)
#else
#define AMP_UNROLL
#endif

namespace amp {

enum { OP_M = 0, OP_I = 1, OP_D = 2, OP_N = 3, OP_S = 4, OP_H = 5, OP_P = 6, OP_EQ = 7, OP_X = 8 };

// AmpliPy.py:43-44 as bit masks over the op code
AMP_HD bool cons_q(uint32_t op) { return (0x193u >> op) & 1u; }   // M I S = X
AMP_HD bool cons_r(uint32_t op) { return (0x18Du >> op) & 1u; }   // M D N = X
AMP_HD bool cons_qr(uint32_t op) { return (0x181u >> op) & 1u; }  // M = X
AMP_HD uint32_t c_op(uint32_t w) { return w & 15u; }
AMP_HD int c_len(uint32_t w) { return (int)(w >> 4); }
AMP_HD uint32_t c_pack(uint32_t op, int n) { return ((uint32_t)n << 4) | op; }

// ---- atomics: real on the device, plain on the host emulation -----------------------------------
AMP_HD int atomic_add(int* p, int v) {
#ifdef __CUDA_ARCH__
    return atomicAdd(p, v);
#else
    int o = *p; *p += v; return o;
#endif
}
AMP_HD unsigned long long atomic_add64(unsigned long long* p, unsigned long long v) {
#ifdef __CUDA_ARCH__
    return atomicAdd(p, v);
#else
    unsigned long long o = *p; *p += v; return o;
#endif
}
// The two cursors of the insertion table (arena words, entry index) are single addresses that every SM hits while the
// generic phases run: lanes of a warp that arrive together combine their requests into one atomic.
AMP_HD unsigned long long atomic_add64_warp(unsigned long long* p, unsigned long long v) {
#ifdef __CUDA_ARCH__
    const unsigned m = __activemask();
    const int lane = (int)(threadIdx.x & 31u), leader = __ffs((int)m) - 1;
    unsigned long long pre = 0, tot = 0;
    for (unsigned r = m; r; r &= r - 1u) {     // (summing the requests a bit plane at a time with ballots measured slower: 1.25 vs 1.09 ms on the ONT batch)
        const int l = __ffs((int)r) - 1;
        const unsigned long long x = __shfl_sync(m, v, l);
        if (l < lane) pre += x;
        tot += x;
    }
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(p, tot);
    base = __shfl_sync(m, base, leader);
    return base + pre;
#else
    unsigned long long o = *p; *p += v; return o;
#endif
}
AMP_HD unsigned long long atomic_cas64(unsigned long long* p, unsigned long long cmp, unsigned long long val) {
#ifdef __CUDA_ARCH__
    return atomicCAS(p, cmp, val);
#else
    unsigned long long o = *p; if (o == cmp) *p = val; return o;
#endif
}
AMP_HD int atomic_cas(int* p, int cmp, int val) {
#ifdef __CUDA_ARCH__
    return atomicCAS(p, cmp, val);
#else
    int o = *p; if (o == cmp) *p = val; return o;
#endif
}
AMP_HD void atomic_min(int* p, int v) {
#ifdef __CUDA_ARCH__
    atomicMin(p, v);
#else
    if (v < *p) *p = v;
#endif
}
AMP_HD void atomic_max(int* p, int v) {
#ifdef __CUDA_ARCH__
    atomicMax(p, v);
#else
    if (v > *p) *p = v;
#endif
}
AMP_HD int atomic_exch(int* p, int v) {
#ifdef __CUDA_ARCH__
    return atomicExch(p, v);
#else
    int o = *p; *p = v; return o;
#endif
}
AMP_HD void atomic_or(unsigned int* p, unsigned int v) {
#ifdef __CUDA_ARCH__
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
AMP_HD void fence() {
#ifdef __CUDA_ARCH__
    __threadfence();
#endif
}
// L1-bypassing loads for data other SMs may have just published (arena records, table keys)
AMP_HD unsigned long long ld_cg64(const unsigned long long* p) {
#ifdef __CUDA_ARCH__
    return __ldcg(p);
#else
    return *p;
#endif
}
AMP_HD unsigned int ld_cg32(const unsigned int* p) {
#ifdef __CUDA_ARCH__
    return __ldcg(p);
#else
    return *p;
#endif
}

// ---- CIGAR helpers on packed ops ---------------------------------------------------------------
AMP_HD int get_pos_on_ref(const uint32_t* c, int nc, int query_pos, int ref_start) {   // 363-386
    int cur = 0, ref_pos = ref_start;
    for (int k = 0; k < nc; ++k) {
        uint32_t op = c_op(c[k]); int n = c_len(c[k]);
        if (cons_q(op)) {
            if (query_pos <= cur + n) { if (cons_r(op)) ref_pos += query_pos - cur; return ref_pos; }
            cur += n;
        }
        if (cons_r(op)) ref_pos += n;
    }
    return ref_pos;
}
AMP_HD int get_pos_on_query(const uint32_t* c, int nc, int ref_pos, int ref_start) {   // 389-412
    int qp = 0, cur = ref_start;
    for (int k = 0; k < nc; ++k) {
        uint32_t op = c_op(c[k]); int n = c_len(c[k]);
        if (cons_r(op)) {
            if (ref_pos <= cur + n) { if (cons_q(op)) qp += ref_pos - cur; return qp; }
            cur += n;
        }
        if (cons_q(op)) qp += n;
    }
    return qp;
}
// htslib bam_endpos floor of 1
AMP_HD int ref_len_of(const uint32_t* c, int nc) {
    int r = 0;
    for (int k = 0; k < nc; ++k) if (cons_r(c_op(c[k]))) r += c_len(c[k]);
    return r == 0 ? 1 : r;
}
AMP_HD int q_align_start(const uint32_t* c, int nc) {
    int s = 0;
    for (int k = 0; k < nc; ++k) {
        uint32_t op = c_op(c[k]);
        if (op == OP_H) continue;
        if (op == OP_S) s += c_len(c[k]); else break;
    }
    return s;
}
AMP_HD int q_align_end(const uint32_t* c, int nc, int l_seq) {
    int e = l_seq;
    for (int k = nc - 1; k >= 1; --k) {   // op 0 is never inspected (pysam getQueryEnd)
        uint32_t op = c_op(c[k]);
        if (op == OP_H) continue;
        if (op == OP_S) e -= c_len(c[k]); else break;
    }
    return e;
}
// append with fix_cigar's merge of equal neighbours (415-423) folded in
AMP_HD void push_op(uint32_t* d, int& nd, uint32_t op, int n) {
    if (nd > 0 && c_op(d[nd - 1]) == op) d[nd - 1] += ((uint32_t)n << 4);
    else d[nd++] = c_pack(op, n);
}
AMP_HD void reverse_ops(uint32_t* d, int nd) {
    for (int i = 0, j = nd - 1; i < j; ++i, --j) { uint32_t t = d[i]; d[i] = d[j]; d[j] = t; }
}

struct TrimParams {
    int L;
    const int32_t* min_primer_start;   // [L], -1 = uncovered   (find_overlapping_primers, 174-209)
    const int32_t* max_primer_end;     // [L], -1 = uncovered
    int max_primer_len, min_quality, window, min_length, include_no_primer;
};

// shared tail of the primer rewrite loops (467-510 and 524-555): one op, forward or reversed order
AMP_HD void primer_rewrite_op(uint32_t w, int& del_len, int& pos_start, int& start_pos, uint32_t* d, int& nd) {
    uint32_t cig = c_op(w); int n = c_len(w);
    if (del_len == 0 && pos_start) { push_op(d, nd, cig, n); return; }
    if (del_len == 0 && cons_qr(cig)) { pos_start = 1; push_op(d, nd, cig, n); return; }
    int ref_add = 0;
    if (cons_q(cig)) {
        if (del_len >= n) push_op(d, nd, OP_S, n);
        else if (0 < del_len && del_len < n) push_op(d, nd, OP_S, del_len);
        else { push_op(d, nd, OP_S, n); return; }
        ref_add = del_len < n ? del_len : n;
        int tmp = n;
        n = (n - del_len) > 0 ? (n - del_len) : 0;
        del_len = (del_len - tmp) > 0 ? (del_len - tmp) : 0;
        uint32_t last = OP_S;
        if (n > 0) { push_op(d, nd, cig, n); last = cig; }
        if (del_len == 0 && cons_qr(last)) pos_start = 1;
    } else if (cons_r(cig)) {
        ref_add += n;
    }
    if (cons_r(cig)) start_pos += ref_add;
}
// quality rewrite loops (597-622 and 658-683): one op
AMP_HD void qual_rewrite_op(uint32_t w, int& del_len, uint32_t* d, int& nd) {
    uint32_t cig = c_op(w); int n = c_len(w);
    if (del_len == 0) { push_op(d, nd, cig, n); return; }
    if (cig == OP_S || cig == OP_H) { push_op(d, nd, cig, n); return; }
    if (cons_q(cig)) {
        if (del_len >= n) push_op(d, nd, OP_S, n); else push_op(d, nd, OP_S, del_len);
        int tmp = n;
        n = (n - del_len) > 0 ? (n - del_len) : 0;
        del_len = (del_len - tmp) > 0 ? (del_len - tmp) : 0;
        if (n > 0) push_op(d, nd, cig, n);
    }
}

// Sliding-window search (closed form of 566-587 / 628-649, verified against the literal loops of
// oracle/amplipy_oracle.c): q = aligned qualities [0, len).  Returns del_len.
//   forward : first i with sum(q[i:i+w]) < minq*w, w = min(W, len-i)  -> len - i   (0 if none)
//   reverse : first i from len down to 1 with sum(q[i-w:i]) < minq*w, w = min(W, i) -> i (0 if none)
AMP_HD int window_del_len_fwd(const uint8_t* q, int len, int W, int minq) {
    if (len <= 0) return 0;
    int w = W < len ? W : len;
    int total = 0;
    for (int j = 0; j < w; ++j) total += q[j];
    for (int i = 0; i < len; ++i) {
        // window [i, i+w)
        if (total < minq * w) return len - i;
        total -= q[i];
        if (i + w < len) total += q[i + w]; else --w;
    }
    return 0;
}
AMP_HD int window_del_len_rev(const uint8_t* q, int len, int W, int minq) {
    if (len <= 0) return 0;
    int w = W < len ? W : len;
    int total = 0;
    for (int j = 0; j < w; ++j) total += q[len - 1 - j];
    for (int i = len; i > 0; --i) {
        // window [i-w, i)
        if (total < minq * w) return i;
        total -= q[i - 1];
        if (i - 1 - w >= 0) total += q[i - 1 - w]; else --w;
    }
    return 0;
}

// ---- word-at-a-time window search for the default width 4 ----------------------------------------
AMP_HD unsigned funnel_r(unsigned lo, unsigned hi, unsigned sh) {   // low 32 bits of (hi:lo) >> (sh & 31)
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    sh &= 31u;
    return sh ? (lo >> sh) | (hi << (32u - sh)) : lo;
#endif
}
AMP_HD unsigned byte_perm(unsigned x, unsigned sel) {               // bytes of x picked by the nibbles of sel
#ifdef __CUDA_ARCH__
    return __byte_perm(x, 0u, sel);
#else
    unsigned r = 0;
    for (int i = 0; i < 4; ++i) r |= ((x >> (8u * ((sel >> (4 * i)) & 3u))) & 0xFFu) << (8 * i);
    return r;
#endif
}
AMP_HD int sum4(unsigned w) {                                       // sum of the four bytes of w
#ifdef __CUDA_ARCH__
    return (int)__dp4a(w, 0x01010101u, 0u);
#else
    return (int)((w & 0xFF) + ((w >> 8) & 0xFF) + ((w >> 16) & 0xFF) + (w >> 24));
#endif
}
AMP_HD unsigned funnel_l(unsigned lo, unsigned hi, unsigned sh) {   // high 32 bits of (hi:lo) << sh, sh in [0, 31]
#ifdef __CUDA_ARCH__
    return __funnelshift_l(lo, hi, sh);
#else
    return sh ? (hi << sh) | (lo >> (32u - sh)) : hi;
#endif
}
AMP_HD unsigned dp4a_acc(unsigned w, unsigned acc) {                // acc + sum of the four bytes of w
#ifdef __CUDA_ARCH__
    return __dp4a(w, 0x01010101u, acc);
#else
    return acc + (w & 0xFF) + ((w >> 8) & 0xFF) + ((w >> 16) & 0xFF) + (w >> 24);
#endif
}
AMP_HD int ctz32(unsigned x) {
#ifdef __CUDA_ARCH__
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
AMP_HD int msb32(unsigned x) {
#ifdef __CUDA_ARCH__
    return 31 - __clz((int)x);
#else
    return 31 - __builtin_clz(x);
#endif
}

// ---- block-wise window search for the default width 4 ---------------------------------------------------------------
// (sum - 4*minq) of the 8 windows starting in read-relative words u0, u1 (u2 = look-ahead): sign bit set = window fails
#define AMP7_WIN8(D, u0, u1, u2, nthr)                                                                              \
    const unsigned D##0 = dp4a_acc(u0, nthr), D##1 = dp4a_acc(funnel_r(u0, u1, 8), nthr),                           \
                   D##2 = dp4a_acc(funnel_r(u0, u1, 16), nthr), D##3 = dp4a_acc(funnel_r(u0, u1, 24), nthr),        \
                   D##4 = dp4a_acc(u1, nthr), D##5 = dp4a_acc(funnel_r(u1, u2, 8), nthr),                           \
                   D##6 = dp4a_acc(funnel_r(u1, u2, 16), nthr), D##7 = dp4a_acc(funnel_r(u1, u2, 24), nthr)
AMP_HD unsigned win8_bits(unsigned u0, unsigned u1, unsigned u2, unsigned nthr) {   // bit w = window w of the block fails
    AMP7_WIN8(D, u0, u1, u2, nthr);
    unsigned F = funnel_l(D7, 0u, 1);
    F = funnel_l(D6, F, 1); F = funnel_l(D5, F, 1); F = funnel_l(D4, F, 1);
    F = funnel_l(D3, F, 1); F = funnel_l(D2, F, 1); F = funnel_l(D1, F, 1); F = funnel_l(D0, F, 1);
    return F;
}
// Sliding-window search (closed form of AmpliPy.py:566-587 / 628-649, same result as window_del_len_fwd / _rev with W = 4)
// for m >= 8, m + (a0 & 3) <= 256: one pass over blocks of 8 windows keeps one "some window fails" bit per block; the
// first (forward strand) / last (reverse strand) failing block is then resolved exactly; the three shrinking windows at
// the open end are checked from three bytes.
AMP_HD int window_del_blocks(const uint8_t* buf, int a0, int m, bool rev, int minq) {
    const uint32_t* A = (const uint32_t*)(buf + (a0 & ~3));
    const unsigned sh = (unsigned)(a0 & 3) << 3;
    const unsigned nthr = (unsigned)(-4 * minq);
    const int nwin = m - 3;                       // full windows start at 0 .. nwin - 1
    const int nb = (nwin + 7) >> 3;               // blocks of 8 windows (<= 32)
    const unsigned last_mask = (1u << (nwin - 8 * (nb - 1))) - 1u;   // valid windows of the last block (1 .. 8 of them)
    unsigned Fw = 0;
    unsigned prev = A[1];
    unsigned u0 = funnel_r(A[0], prev, sh);
#if defined(__CUDA_ARCH__) && defined(AMP_WINDOW_UNROLL)
    AMP_UNROLL_N(AMP_WINDOW_UNROLL)
#endif
    for (int i = 0; i < nb - 1; ++i) {
        const unsigned x1 = A[2 * i + 2], x2 = A[2 * i + 3];
        const unsigned u1 = funnel_r(prev, x1, sh), u2 = funnel_r(x1, x2, sh);
        AMP7_WIN8(D, u0, u1, u2, nthr);
        Fw = funnel_l(D0 | D1 | D2 | D3 | D4 | D5 | D6 | D7, Fw, 1);
        u0 = u2; prev = x2;
    }
    {
        const unsigned x1 = A[2 * nb], x2 = A[2 * nb + 1];
        const unsigned bits = win8_bits(u0, funnel_r(prev, x1, sh), funnel_r(x1, x2, sh), nthr) & last_mask;
        Fw = (Fw << 1) | (bits ? 1u : 0u);
    }
    if (Fw) {   // block i sits at bit nb - 1 - i
        const int i = nb - 1 - (rev ? ctz32(Fw) : msb32(Fw));
        const unsigned x0 = A[2 * i], x1 = A[2 * i + 1], x2 = A[2 * i + 2], x3 = A[2 * i + 3];
        unsigned bits = win8_bits(funnel_r(x0, x1, sh), funnel_r(x1, x2, sh), funnel_r(x2, x3, sh), nthr);
        if (i == nb - 1) bits &= last_mask;
        const int t = 8 * i + (rev ? msb32(bits) : ctz32(bits));
        return rev ? t + 4 : m - t;
    }
    const uint8_t* e3 = buf + a0 + (rev ? 0 : m - 3);   // shrinking windows w = 3, 2, 1 at the open end
    const int x0 = e3[0], x1 = e3[1], x2 = e3[2];
    const int e = rev ? x0 : x2;
    if (x0 + x1 + x2 < 3 * minq) return 3;
    if (e + x1 < 2 * minq) return 2;
    if (e < minq) return 1;
    return 0;
}

// Same result as window_del_len_fwd / _rev for W == 4, scanning the logical sequence s[t] = rev ? q[len-1-t] : q[t]
// four positions per step (one aligned word + funnel shifts + dp4a), identical instruction stream for both
// strands.  Requires 8 readable bytes before and 16 after q[0, len) (true inside the staging buffers).
AMP_HD int window_del_len_w4(const uint8_t* q, int len, int minq, bool rev) {
    {   // common case: the block-wise search (16 readable bytes after the run)
        const int mis = (int)((uintptr_t)q & 3u);
        if (len >= 8 && mis + len <= 256) return window_del_blocks(q - mis, mis, len, rev, minq);
    }
    const int thr = 4 * minq;
    int t = 0;
    if (len >= 7) {
        const uint8_t* a0 = rev ? q + len - 4 : q;
        const unsigned sh = (unsigned)((uintptr_t)a0 & 3u) * 8u;
        const uint32_t* wp = (const uint32_t*)(a0 - ((uintptr_t)a0 & 3u));
        const int wstep = rev ? -1 : 1;
        const unsigned sel = rev ? 0x0123u : 0x3210u;
        const int ngroups = (len - 7) / 4 + 1;
        unsigned v0 = byte_perm(funnel_r(wp[0], wp[1], sh), sel);
        for (int g = 0; g < ngroups; ++g) {
            wp += wstep;
            const unsigned v1 = byte_perm(funnel_r(wp[0], wp[1], sh), sel);
            const int s0 = sum4(v0), s1 = sum4(funnel_r(v0, v1, 8)), s2 = sum4(funnel_r(v0, v1, 16)), s3 = sum4(funnel_r(v0, v1, 24));
            int m = s0 < s1 ? s0 : s1; const int m2 = s2 < s3 ? s2 : s3; m = m < m2 ? m : m2;
            if (m < thr) return len - (4 * g + (s0 < thr ? 0 : s1 < thr ? 1 : s2 < thr ? 2 : 3));
            v0 = v1;
        }
        t = 4 * ngroups;
    }
    return rev ? window_del_len_rev(q, len - t, 4, minq) : window_del_len_fwd(q + t, len - t, 4, minq);
}

// Both strands of the sliding-window search in one loop: with s[t] = rev ? q[len-1-t] : q[t], window_del_len_fwd and
// window_del_len_rev are the same scan over t and both return len - t at the first failing window.  Lanes of a warp
// working on reads of either strand stay together in it.
AMP_HD int window_del_len_any(const uint8_t* q, int len, int W, int minq, bool rev) {
    if (len <= 0) return 0;
    const int step = rev ? -1 : 1;
    const uint8_t* s = rev ? q + len - 1 : q;
    int w = W < len ? W : len;
    int total = 0;
    for (int j = 0; j < w; ++j) total += s[j * step];
    for (int t = 0; t < len; ++t) {
        if (total < minq * w) return len - t;
        total -= s[t * step];
        if (t + w < len) total += s[(t + w) * step]; else --w;
    }
    return 0;
}

// trim_read (426-687).  A holds the input CIGAR (capacity nc+3), B is scratch of the same capacity.
// On return *res points at the buffer holding the final CIGAR.  Returns AMP_F_* bits.
// qual_padded: the qualities sit in a staging buffer with readable slack around them (enables the word-wise search).
// lanes != 0 (device, lane-per-read callers): the mask of lanes that entered together; they are brought together again
// after each of the three steps, whose loops otherwise drift apart for the rest of the read (every lane named in the
// mask passes every one of these points: the coordinate check only marks the read as bad instead of returning early).
AMP_HD int trim_read(uint32_t* A, uint32_t* B, int& nc, int& pos, int flag, int tlen, int l_seq, const uint8_t* qual,
                     bool qual_padded, const TrimParams& P, uint32_t** res, unsigned lanes = 0) {
#ifdef __CUDA_ARCH__
#define AMP_TR_SYNC() do { if (lanes) __syncwarp(lanes); } while (0)
#else
#define AMP_TR_SYNC() ((void)lanes)
#endif
    uint32_t* src = A; uint32_t* dst = B;
    int ref_start = pos;
    const bool is_paired = flag & 1, is_reverse = (flag & 16) != 0;
    int ref_end = ref_start + ref_len_of(src, nc);
    *res = src;
    const bool bad = ref_start < 0 || ref_start >= P.L || ref_end - 1 >= P.L;
    if (bad && !lanes) return AMP_F_ERROR;
    const int left_max_primer_end = bad ? -1 : P.max_primer_end[ref_start];        // 450
    const int right_min_primer_start = bad ? -1 : P.min_primer_start[ref_end - 1];  // 451
    const int abs_tlen = tlen < 0 ? -tlen : tlen;
    const bool isize_flag = (abs_tlen - P.max_primer_len) > l_seq;       // 452
    int out = 0;

    if (!(is_paired && isize_flag && is_reverse) && left_max_primer_end >= 0) {          // 460
        out |= AMP_F_TRIM_START;
        int del_len = get_pos_on_query(src, nc, left_max_primer_end + 1, ref_start);     // 463
        int nd = 0, pos_start = 0, start_pos = 0;
        for (int k = 0; k < nc; ++k) primer_rewrite_op(src[k], del_len, pos_start, start_pos, dst, nd);
        nc = nd; { uint32_t* t = src; src = dst; dst = t; }
        ref_start += start_pos;                                                          // 514
    }
    AMP_TR_SYNC();
    if (!(is_paired && isize_flag && !is_reverse) && right_min_primer_start >= 0) {      // 517
        out |= AMP_F_TRIM_END;
        int del_len = l_seq - get_pos_on_query(src, nc, right_min_primer_start, ref_start);   // 520
        int nd = 0, pos_start = 0, dummy = 0;
        for (int k = nc - 1; k >= 0; --k) primer_rewrite_op(src[k], del_len, pos_start, dummy, dst, nd);
        reverse_ops(dst, nd);
        nc = nd; { uint32_t* t = src; src = dst; dst = t; }
    }
    AMP_TR_SYNC();
    const int qas = q_align_start(src, nc);
    int len = q_align_end(src, nc, l_seq) - qas;                                         // 561-563
    if (len < 0) len = 0;
    const bool w4 = qual_padded && P.window == 4;
    // 566-587 (reverse strand) / 628-649 (forward strand)
    const int del_len0 = w4 ? window_del_len_w4(qual + qas, len, P.min_quality, is_reverse)
                            : window_del_len_any(qual + qas, len, P.window, P.min_quality, is_reverse);
    AMP_TR_SYNC();
    // reverse strand: clip from the start iff it moves the first aligned position (591-594); reference_start is NOT
    // advanced (589-625; SURVEY.md F6).  Forward strand: clip from the end iff del_len != 0 (656).
    const bool clip = !bad && (is_reverse ? get_pos_on_ref(src, nc, del_len0 + qas - 1, ref_start) > ref_start : del_len0 != 0);
    if (clip) {
        out |= AMP_F_TRIM_QUAL;
        int del_len = del_len0, nd = 0;
        for (int k = 0; k < nc; ++k) qual_rewrite_op(src[is_reverse ? k : nc - 1 - k], del_len, dst, nd);   // 597-622 / 658-683
        if (!is_reverse) reverse_ops(dst, nd);
        nc = nd; { uint32_t* t = src; src = dst; dst = t; }
    }
    AMP_TR_SYNC();
    if (bad) return AMP_F_ERROR;
    if (ref_len_of(src, nc) >= P.min_length && ((out & (AMP_F_TRIM_START | AMP_F_TRIM_END)) || P.include_no_primer))
        out |= AMP_F_KEEP;                                                               // 910
    pos = ref_start;
    *res = src;
    return out;
#undef AMP_TR_SYNC
}

// ---- register-only fast path for the dominant CIGAR shape [S] M [S] --------------------------------------
// Closed form of trim_read (426-687) for a mapped read whose CIGAR is  S(s1)? (M|=|X)(m) S(s2)?  with
// s1 + m + s2 == l_seq.  Each step is the generic rewrite loop evaluated symbolically for this shape:
//   start  : d1 = max_primer_end[pos] + 1 - pos bases leave the aligned run (one past the primer, 463),
//            pos advances by d1 (514)
//   end    : d2 = reference_end - min_primer_start[reference_end - 1] bases leave it from the right (520)
//   quality: the window search result clips from the right (forward) or from the left WITHOUT moving pos
//            (reverse, 589-625), reverse only when del_len >= 2 (591-594)
// Anything unusual (offset-induced d1 < 1, a primer swallowing the whole run, coordinates outside the genome,
// unstaged qualities) returns false and the caller runs the generic trim_read instead -- so this path never has
// to reproduce the reference's corner cases, only recognise them.
struct SimpleRead { int s1, m, s2; uint32_t mop; };    // mop = op code of the aligned run (0, 7 or 8)
AMP_HD bool classify_simple(const uint32_t* cig, int nc, int l_seq, SimpleRead& r) {
    if (nc < 1 || nc > 3) return false;
    int k = 0;
    r.s1 = 0; r.s2 = 0;
    if (c_op(cig[0]) == OP_S) { r.s1 = c_len(cig[0]); if (r.s1 < 1) return false; k = 1; }
    if (k >= nc || !cons_qr(c_op(cig[k]))) return false;
    r.mop = c_op(cig[k]); r.m = c_len(cig[k]); ++k;
    if (k < nc) { if (c_op(cig[k]) != OP_S) return false; r.s2 = c_len(cig[k]); if (r.s2 < 1) return false; ++k; }
    return k == nc && r.m >= 1 && r.s1 + r.m + r.s2 == l_seq;
}
// the same classification from the first three CIGAR words held in registers (w_k is ignored for k >= nc)
AMP_HD bool classify_simple3(int nc, uint32_t w0, uint32_t w1, uint32_t w2, int l_seq, SimpleRead& r) {
    if (nc < 1 || nc > 3) return false;
    int k = 0;
    r.s1 = 0; r.s2 = 0;
    if (c_op(w0) == OP_S) { r.s1 = c_len(w0); if (r.s1 < 1) return false; k = 1; }
    if (k >= nc) return false;
    const uint32_t mw = k ? w1 : w0;
    if (!cons_qr(c_op(mw))) return false;
    r.mop = c_op(mw); r.m = c_len(mw); ++k;
    if (k < nc) { const uint32_t sw = k == 1 ? w1 : w2; if (c_op(sw) != OP_S) return false; r.s2 = c_len(sw); if (r.s2 < 1) return false; ++k; }
    return k == nc && r.m >= 1 && r.s1 + r.m + r.s2 == l_seq;
}
// Steps 1-2 (primer start / end) of the closed form.  On success r / pos hold the shape after primer clipping.
AMP_HD bool trim_simple_primers(SimpleRead& r, int& pos, int flag, int tlen, int l_seq, const TrimParams& P, int* flags_out) {
    const int p = pos, ref_end = p + r.m;
    if (p < 0 || ref_end > P.L) return false;
    const bool paired = flag & 1, rev = (flag & 16) != 0;
    const int L1 = P.max_primer_end[p];                                   // 450
    const int R1 = P.min_primer_start[ref_end - 1];                       // 451
    const int abs_tlen = tlen < 0 ? -tlen : tlen;
    const bool isize = (abs_tlen - P.max_primer_len) > l_seq;             // 452
    int s1 = r.s1, m = r.m, s2 = r.s2, pp = p, f = 0;
    if (!(paired && isize && rev) && L1 >= 0) {                           // 460
        const int d1 = L1 + 1 - p;
        if (d1 < 1 || d1 >= m) return false;
        f |= AMP_F_TRIM_START; s1 += d1; m -= d1; pp += d1;
    }
    if (!(paired && isize && !rev) && R1 >= 0) {                          // 517
        const int e = R1 - pp;                                            // aligned bases that stay
        if (e < 1 || e >= m) return false;
        f |= AMP_F_TRIM_END; s2 += m - e; m = e;
    }
    r.s1 = s1; r.m = m; r.s2 = s2; pos = pp; *flags_out = f;
    return true;
}
// Step 3 (quality clip, given the window search result `del` over the aligned run) + the write gate (910).
AMP_HD void trim_simple_finish(SimpleRead& r, int del, bool rev, const TrimParams& P, int* flags_io) {
    int f = *flags_io;
    if (rev) { if (del >= 2) { f |= AMP_F_TRIM_QUAL; r.s1 += del; r.m -= del; } }      // pos stays (F6)
    else if (del != 0) { f |= AMP_F_TRIM_QUAL; r.s2 += del; r.m -= del; }
    const int ref_len = r.m > 0 ? r.m : 1;
    if (ref_len >= P.min_length && ((f & (AMP_F_TRIM_START | AMP_F_TRIM_END)) || P.include_no_primer)) f |= AMP_F_KEEP;   // 910
    *flags_io = f;
}
// On success: r = final shape, pos = final reference_start, returns AMP_F_* bits (incl. KEEP) in *flags_out.
AMP_HD bool trim_simple(SimpleRead& r, int& pos, int flag, int tlen, int l_seq, const uint8_t* qual, bool qual_padded,
                        const TrimParams& P, int* flags_out) {
    int f = 0;
    if (!trim_simple_primers(r, pos, flag, tlen, l_seq, P, &f)) return false;
    const bool rev = (flag & 16) != 0;
    const bool w4 = qual_padded && P.window == 4;
    const uint8_t* q = qual + r.s1;
    const int del = w4 ? window_del_len_w4(q, r.m, P.min_quality, rev)
                       : (rev ? window_del_len_rev(q, r.m, P.window, P.min_quality) : window_del_len_fwd(q, r.m, P.window, P.min_quality));
    trim_simple_finish(r, del, rev, P, &f);
    *flags_out = f;
    return true;
}
// final CIGAR of a simple read: [S] [M] [S]; an emptied aligned run leaves one merged soft clip (fix_cigar)
AMP_HD int emit_simple(const SimpleRead& r, uint32_t* out) {
    if (r.m <= 0) { out[0] = c_pack(OP_S, r.s1 + r.s2); return 1; }
    int n = 0;
    if (r.s1 > 0) out[n++] = c_pack(OP_S, r.s1);
    out[n++] = c_pack(r.mop, r.m);
    if (r.s2 > 0) out[n++] = c_pack(OP_S, r.s2);
    return n;
}

// ---- register-only closed form for  [H] [S] M [ (I|D) M ] [S] [H]  ------------------------------------------------------
// The shapes short-read aligners produce for all but a fraction of a percent of the reads: one aligned run or two runs
// around a single insertion / deletion, with optional soft and hard clips.  trim_read (426-687) and update_base_counts
// (690-753) are evaluated symbolically on the seven lengths:
//   primer clips : as for [S]M[S]; they must end strictly inside the outer aligned run on their side, otherwise the closed
//                  form declines and the caller runs the generic trim_read (a hard clip on a clipped side is dropped, 481/505)
//   quality clip : T query bases leave the aligned part from the end (forward) or the start (reverse, pos stays: F6),
//                  whatever they cross: an insertion shrinks base by base (597-622: I -> S), a deletion survives only when the
//                  clip stops exactly at it and is dropped as soon as it is crossed
//   pileup       : up to two aligned runs, one deletion run, and the insertion state machine (730-748) over the k inserted
//                  bases with its exits (A) next pair is a match, (C) next pair is the trailing clip, (D) low-quality base
struct Shape5 {
    int h1, s1, m, k, m2, s2, h2;   // lengths; k = 0: no indel left; m / m2 may reach 0 by clipping
    uint32_t ops;                   // op code of the first run | of the second run << 4 | OP_I or OP_D << 8
};
AMP_HD uint32_t shape_xop(const Shape5& r) { return (r.ops >> 8) & 15u; }
AMP_HD bool shape_is_ins(const Shape5& r) { return r.k > 0 && shape_xop(r) == OP_I; }
AMP_HD bool shape_is_del(const Shape5& r) { return r.k > 0 && shape_xop(r) == OP_D; }
AMP_HD int shape_qlen(const Shape5& r) { return r.m + r.m2 + (shape_is_ins(r) ? r.k : 0); }      // aligned query bases
AMP_HD int shape_rlen(const Shape5& r) { return r.m + r.m2 + (shape_is_del(r) ? r.k : 0); }      // reference bases
// classification from the first five CIGAR words held in registers (w_k is ignored for k >= nc)
AMP_HD bool classify_shape5(int nc, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t w4, int l_seq, Shape5& r) {
    r.h1 = r.s1 = r.m = r.k = r.m2 = r.s2 = r.h2 = 0; r.ops = 0;
    if (nc < 1 || nc > 5) return false;
    if (nc < 5) w4 = 15u;            // op 15 matches nothing
    if (nc < 4) w3 = 15u;
    if (nc < 3) w2 = 15u;
    if (nc < 2) w1 = 15u;
    int used = 0;
#define AMP_POP() do { w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = 15u; ++used; } while (0)
    if (c_op(w0) == OP_H) { r.h1 = c_len(w0); if (r.h1 < 1) return false; AMP_POP(); }
    if (c_op(w0) == OP_S) { r.s1 = c_len(w0); if (r.s1 < 1) return false; AMP_POP(); }
    if (!cons_qr(c_op(w0))) return false;
    r.ops = c_op(w0); r.m = c_len(w0); if (r.m < 1) return false; AMP_POP();
    if (c_op(w0) == OP_I || c_op(w0) == OP_D) {
        r.ops |= c_op(w0) << 8; r.k = c_len(w0); if (r.k < 1) return false; AMP_POP();
        if (!cons_qr(c_op(w0))) return false;
        r.ops |= c_op(w0) << 4; r.m2 = c_len(w0); if (r.m2 < 1) return false; AMP_POP();
    }
    if (c_op(w0) == OP_S) { r.s2 = c_len(w0); if (r.s2 < 1) return false; AMP_POP(); }
    if (c_op(w0) == OP_H) { r.h2 = c_len(w0); if (r.h2 < 1) return false; AMP_POP(); }
#undef AMP_POP
    return used == nc && r.s1 + shape_qlen(r) + r.s2 == l_seq;
}
// Steps 1-2 (primer start / end).  On success r / pos hold the shape after primer clipping.
AMP_HD bool trim_shape_primers(Shape5& r, int& pos, int flag, int tlen, int l_seq, const TrimParams& P, int* flags_out) {
    const int gap = shape_is_del(r) ? r.k : 0;
    const int p = pos, ref_end = p + r.m + gap + r.m2;
    if (p < 0 || ref_end > P.L) return false;
    const bool paired = flag & 1, rev = (flag & 16) != 0;
    const int L1 = P.max_primer_end[p];                                   // 450
    const int R1 = P.min_primer_start[ref_end - 1];                       // 451
    const int abs_tlen = tlen < 0 ? -tlen : tlen;
    const bool isize = (abs_tlen - P.max_primer_len) > l_seq;             // 452
    int pp = p, f = 0;
    if (!(paired && isize && rev) && L1 >= 0) {                           // 460
        const int d1 = L1 + 1 - p;                                        // one base past the primer (463)
        if (d1 < 1) return false;
        if (d1 < r.m) { r.s1 += d1; r.m -= d1; pp += d1; }
        else {
            // the clip crosses the indel (467-510): an insertion inside the clipped span becomes soft clip (487-488 when the
            // clip ends exactly in front of it), a deletion is dropped and the start advances over it (quirk table, SURVEY 8a-Q);
            // d more bases leave the second run, which is all that remains
            if (r.k == 0) return false;
            const int d = gap ? (d1 - r.m - gap > 0 ? d1 - r.m - gap : 0) : d1 - r.m;
            if (d >= r.m2) return false;
            r.s1 += r.m + (gap ? 0 : r.k) + d; pp += r.m + gap + d;
            r.m = r.m2 - d; r.ops = (r.ops >> 4) & 15u; r.k = 0; r.m2 = 0;
        }
        f |= AMP_F_TRIM_START; r.h1 = 0;
    }
    if (!(paired && isize && !rev) && R1 >= 0) {                          // 517
        const int gap2 = shape_is_del(r) ? r.k : 0;
        if (r.k > 0 && R1 > pp + r.m + gap2) {
            const int e = R1 - (pp + r.m + gap2);                         // bases of the second run that stay
            if (e >= r.m2) return false;
            r.s2 += r.m2 - e; r.m2 = e;
        } else {
            // inside the only run -- or, across the indel, inside the first run (524-555 over the reversed ops: the inserted
            // bases turn into soft clip, a deletion is dropped; a target inside the deletion keeps the whole first run)
            int e = R1 - pp;                                              // aligned bases that stay
            if (e < 1) return false;
            if (r.k > 0) { if (e > r.m) e = r.m; r.k = 0; r.m2 = 0; r.ops &= 15u; }
            else if (e >= r.m) return false;
            r.m = e; r.s2 = l_seq - r.s1 - e;
        }
        f |= AMP_F_TRIM_END; r.h2 = 0;
    }
    pos = pp; *flags_out = f;
    return true;
}
// Step 3 (quality clip, given the window search result `del` over the aligned query bases) + the write gate (910).
AMP_HD void trim_shape_finish(Shape5& r, int del, bool rev, const TrimParams& P, int* flags_io) {
    int f = *flags_io;
    if (rev ? del >= 2 : del != 0) {                                      // 591-594 / 656
        f |= AMP_F_TRIM_QUAL;
        const bool is_ins = shape_is_ins(r);
        int T = del;
        if (rev) {                                                        // from the start; pos stays (F6)
            r.s1 += T;
            if (T < r.m) r.m -= T;
            else {
                T -= r.m; r.m = 0;
                if (r.k > 0) {
                    if (is_ins) { if (T < r.k) { r.k -= T; T = 0; } else { T -= r.k; r.k = 0; } }
                    else if (T > 0) r.k = 0;                              // a crossed deletion is dropped
                }
                r.m2 -= T;
            }
        } else {                                                          // from the end
            r.s2 += T;
            if (T < r.m2) r.m2 -= T;
            else {
                T -= r.m2; r.m2 = 0;
                if (r.k > 0) {
                    if (is_ins) { if (T < r.k) { r.k -= T; T = 0; } else { T -= r.k; r.k = 0; } }
                    else if (T > 0) r.k = 0;
                }
                r.m -= T;
            }
        }
        if (r.m <= 0 && r.k == 0 && r.m2 > 0) { r.m = r.m2; r.m2 = 0; r.ops = (r.ops & ~15u) | ((r.ops >> 4) & 15u); }
    }
    const int rl = shape_rlen(r);
    const int ref_len = rl > 0 ? rl : 1;
    if (ref_len >= P.min_length && ((f & (AMP_F_TRIM_START | AMP_F_TRIM_END)) || P.include_no_primer)) f |= AMP_F_KEEP;   // 910
    *flags_io = f;
}
// final CIGAR; an emptied aligned part leaves one merged soft clip (fix_cigar)
AMP_HD int emit_shape5(const Shape5& r, uint32_t* out) {
    int n = 0;
    if (r.h1 > 0) out[n++] = c_pack(OP_H, r.h1);
    if (r.m <= 0 && r.k <= 0 && r.m2 <= 0) out[n++] = c_pack(OP_S, r.s1 + r.s2);
    else {
        if (r.s1 > 0) out[n++] = c_pack(OP_S, r.s1);
        if (r.m > 0) out[n++] = c_pack(r.ops & 15u, r.m);
        if (r.k > 0) out[n++] = c_pack(shape_xop(r), r.k);
        if (r.m2 > 0) out[n++] = c_pack((r.ops >> 4) & 15u, r.m2);
        if (r.s2 > 0) out[n++] = c_pack(OP_S, r.s2);
    }
    if (r.h2 > 0) out[n++] = c_pack(OP_H, r.h2);
    return n;
}
// the insertion alleles of the final shape (730-748); emit(pos, first base, length) as plan_read's sink.ins.
// qual = the read's qualities (query index 0 at qual[0]).
template <class Emit>
AMP_HD void shape_ins_events(const Shape5& r, int pos, int l_seq, const uint8_t* qual, int minq, Emit& emit) {
    if (!shape_is_ins(r)) return;
    const int qI = r.s1 + r.m, rI = pos + r.m, qend = qI + r.k;
    const int rl = r.m + r.m2;
    int anchor = pos + (rl > 0 ? rl : 1) - 1; if (anchor < 0) anchor = 0;        // max(reference_end - 1, 0)
    int q0 = -1;
    for (int j = qI; j < qend; ++j) {
        const bool pass = qual[j] >= minq;
        if (q0 < 0) { if (pass) q0 = j; }                                        // 718 / 732
        else if (!pass) { emit(anchor, q0 - 1, j - (q0 - 1)); q0 = -1; }         // exit (D)
    }
    if (q0 < 0) return;
    if (r.m2 > 0) {                                                              // exit (A) / (A')
        if (rI == 0) { const int e = qend + 1 < l_seq ? qend + 1 : l_seq; emit(0, q0, e - q0); }
        else emit(rI - 1, q0 - 1, qend - (q0 - 1));
    } else emit(anchor, q0 - 1, qend - (q0 - 1));                                // exit (C): the trailing clip follows
}

// ---- sequence access: BAM 4-bit nibbles, high nibble first ---------------------------------------
AMP_HD uint32_t nib_at(const uint8_t* seq, uint32_t idx) { return (seq[idx >> 1] >> ((~idx & 1u) << 2)) & 15u; }
AMP_HD char nib_char(uint32_t nib) {
    // "=ACMGRSVTWYHKDBN"
#ifdef __CUDA_ARCH__
    const unsigned lo = __byte_perm(0x4D43413Du, 0x56535247u, nib & 7u);   // byte (nib & 7) of "=ACMGRSV"
    const unsigned hi = __byte_perm(0x48595754u, 0x4E42444Bu, nib & 7u);   // ... of "TWYHKDBN"
    return (char)((nib & 8u ? hi : lo) & 0xFFu);
#else
    const unsigned long long lo = 0x565352474D43413DULL;  // "=ACMGRSV" little-endian bytes
    const unsigned long long hi = 0x4E42444B48595754ULL;  // "TWYHKDBN"
    return (char)(((nib < 8 ? lo : hi) >> ((nib & 7u) * 8u)) & 0xFFu);
#endif
}
// one packed byte -> the characters of its two bases (first base in the low byte): 256 x u16, constant memory on the device
#define AMP_NIBPAIR_INIT \
    0x3D3D, 0x413D, 0x433D, 0x4D3D, 0x473D, 0x523D, 0x533D, 0x563D, 0x543D, 0x573D, 0x593D, 0x483D, 0x4B3D, 0x443D, 0x423D, 0x4E3D, \
    0x3D41, 0x4141, 0x4341, 0x4D41, 0x4741, 0x5241, 0x5341, 0x5641, 0x5441, 0x5741, 0x5941, 0x4841, 0x4B41, 0x4441, 0x4241, 0x4E41, \
    0x3D43, 0x4143, 0x4343, 0x4D43, 0x4743, 0x5243, 0x5343, 0x5643, 0x5443, 0x5743, 0x5943, 0x4843, 0x4B43, 0x4443, 0x4243, 0x4E43, \
    0x3D4D, 0x414D, 0x434D, 0x4D4D, 0x474D, 0x524D, 0x534D, 0x564D, 0x544D, 0x574D, 0x594D, 0x484D, 0x4B4D, 0x444D, 0x424D, 0x4E4D, \
    0x3D47, 0x4147, 0x4347, 0x4D47, 0x4747, 0x5247, 0x5347, 0x5647, 0x5447, 0x5747, 0x5947, 0x4847, 0x4B47, 0x4447, 0x4247, 0x4E47, \
    0x3D52, 0x4152, 0x4352, 0x4D52, 0x4752, 0x5252, 0x5352, 0x5652, 0x5452, 0x5752, 0x5952, 0x4852, 0x4B52, 0x4452, 0x4252, 0x4E52, \
    0x3D53, 0x4153, 0x4353, 0x4D53, 0x4753, 0x5253, 0x5353, 0x5653, 0x5453, 0x5753, 0x5953, 0x4853, 0x4B53, 0x4453, 0x4253, 0x4E53, \
    0x3D56, 0x4156, 0x4356, 0x4D56, 0x4756, 0x5256, 0x5356, 0x5656, 0x5456, 0x5756, 0x5956, 0x4856, 0x4B56, 0x4456, 0x4256, 0x4E56, \
    0x3D54, 0x4154, 0x4354, 0x4D54, 0x4754, 0x5254, 0x5354, 0x5654, 0x5454, 0x5754, 0x5954, 0x4854, 0x4B54, 0x4454, 0x4254, 0x4E54, \
    0x3D57, 0x4157, 0x4357, 0x4D57, 0x4757, 0x5257, 0x5357, 0x5657, 0x5457, 0x5757, 0x5957, 0x4857, 0x4B57, 0x4457, 0x4257, 0x4E57, \
    0x3D59, 0x4159, 0x4359, 0x4D59, 0x4759, 0x5259, 0x5359, 0x5659, 0x5459, 0x5759, 0x5959, 0x4859, 0x4B59, 0x4459, 0x4259, 0x4E59, \
    0x3D48, 0x4148, 0x4348, 0x4D48, 0x4748, 0x5248, 0x5348, 0x5648, 0x5448, 0x5748, 0x5948, 0x4848, 0x4B48, 0x4448, 0x4248, 0x4E48, \
    0x3D4B, 0x414B, 0x434B, 0x4D4B, 0x474B, 0x524B, 0x534B, 0x564B, 0x544B, 0x574B, 0x594B, 0x484B, 0x4B4B, 0x444B, 0x424B, 0x4E4B, \
    0x3D44, 0x4144, 0x4344, 0x4D44, 0x4744, 0x5244, 0x5344, 0x5644, 0x5444, 0x5744, 0x5944, 0x4844, 0x4B44, 0x4444, 0x4244, 0x4E44, \
    0x3D42, 0x4142, 0x4342, 0x4D42, 0x4742, 0x5242, 0x5342, 0x5642, 0x5442, 0x5742, 0x5942, 0x4842, 0x4B42, 0x4442, 0x4242, 0x4E42, \
    0x3D4E, 0x414E, 0x434E, 0x4D4E, 0x474E, 0x524E, 0x534E, 0x564E, 0x544E, 0x574E, 0x594E, 0x484E, 0x4B4E, 0x444E, 0x424E, 0x4E4E
#ifdef __CUDACC__
__device__ __constant__ uint16_t kNibPairDev[256] = {AMP_NIBPAIR_INIT};
#endif
static const uint16_t kNibPairHost[256] = {AMP_NIBPAIR_INIT};
AMP_HD uint32_t nib_pair_chars(uint32_t byte) {
#ifdef __CUDA_ARCH__
    return kNibPairDev[byte & 255u];
#else
    return kNibPairHost[byte & 255u];
#endif
}
// channel of an aligned base: A C G T N -> 0..4, anything else -> -1
AMP_HD int nib_channel(uint32_t nib) {
    switch (nib) { case 1: return 0; case 2: return 1; case 4: return 2; case 8: return 3; case 15: return 4; default: return -1; }
}

// ---- insertion-allele hash table ------------------------------------------------------------------
// slot  : key64 = [tag:24 | arena offset in 8-byte words:40] (0 = empty), count32, next = the position's next allele (-1 = last)
// arena : records {int32 gpos; uint32 len; char text[len]} padded to 8 bytes, write-once
// Lookups compare the full text, so the hash is only a filter: results are exact.
struct InsSlot { unsigned long long key; int count; int next; };
struct InsTable {
    InsSlot* slots; unsigned long long mask;        // capacity - 1 (power of two)
    unsigned int* entries;                           // dense list: entries[k] = slot of the k-th distinct allele
    int* slot_entry;                                 // inverse: slot -> k
    unsigned char* arena; unsigned long long arena_words;
    unsigned long long* cursor;                      // [0] = arena words used, [1] = entries used
    unsigned int* err;
    int* heads;                                      // [n_samples * Lpad] first slot of the position's allele list, -1 = none;
                                                     // null: no lists kept (a table whose user links them when it reads them)
};
AMP_HD unsigned long long mix64(unsigned long long h) {
    h ^= h >> 30; h *= 0xBF58476D1CE4E5B9ULL; h ^= h >> 27; h *= 0x94D049BB133111EBULL; h ^= h >> 31; return h;
}
// text getter: text(i) -> i-th character of the key; text.word(i, len) -> characters i .. i+3 packed little-endian
// (i a multiple of 4, zero beyond len).  Keys are hashed, stored and compared a word at a time: insertion alleles that
// run to the end of the read (exit (B) of the state machine) are hundreds of characters long.
// The key's hash is built from these three steps (ins_table_add interleaves the middle one with writing a long key's record)
AMP_HD unsigned long long ins_hash_init(int gpos) { return (0xCBF29CE484222325ULL ^ (unsigned long long)(unsigned int)gpos) * 0x100000001B3ULL; }
AMP_HD unsigned long long ins_hash_word(unsigned long long h, unsigned int w) { return (h ^ w) * 0x100000001B3ULL; }
AMP_HD unsigned long long ins_hash_final(unsigned long long h, int len) { return mix64(h ^ ((unsigned long long)len << 32)); }
// slot key k (tag matched) names the record of exactly this key
template <class Text>
AMP_HD bool ins_rec_equal(const InsTable& T, unsigned long long k, int gpos, int len, const Text& text) {
    fence();
    const unsigned char* rec = T.arena + (k & 0xFFFFFFFFFFULL) * 8;
    const unsigned long long hdr = ld_cg64((const unsigned long long*)rec);
    if ((int)(hdr & 0xFFFFFFFFu) != gpos || (unsigned int)(hdr >> 32) != (unsigned int)len) return false;
    bool same = true;
    for (int i = 0; i < len && same; i += 4) {
        unsigned int w = ld_cg32((const unsigned int*)(rec + 8 + i));
        if (len - i < 4) w &= (1u << (8 * (len - i))) - 1u;
        same = w == text.word(i, len);
    }
    return same;
}
template <class Text>
AMP_HD_NOINLINE void ins_table_add(const InsTable& T, int gpos, int len, const Text& text, int n) {
    unsigned long long h = ins_hash_init(gpos);
    long long my_off = -1;
#ifndef AMP_KEY_SPEC
#define AMP_KEY_SPEC 32
#endif
    if (len >= AMP_KEY_SPEC) {
        // a key this long is almost always new (an insertion running into a deletion: the rest of the read): its record
        // is written while it is hashed, one pass over the text instead of two; if the allele turns out to be known the
        // record stays behind unused
        const unsigned long long words = 1 + ((unsigned long long)len + 7) / 8;
        const unsigned long long off = atomic_add64_warp(&T.cursor[0], words);
        if (off + words > T.arena_words) { atomic_or(T.err, AMP_E_ARENA_FULL); return; }
        unsigned char* rec = T.arena + off * 8;
        ((int*)rec)[0] = gpos; ((unsigned int*)rec)[1] = (unsigned int)len;
        for (int i = 0; i < len; i += 4) {
            const unsigned int w = text.word(i, len);
            ((unsigned int*)(rec + 8))[i >> 2] = w;
            h = ins_hash_word(h, w);
        }
        fence();
        my_off = (long long)off;
    } else {
        for (int i = 0; i < len; i += 4) h = ins_hash_word(h, text.word(i, len));
    }
    h = ins_hash_final(h, len);
    const unsigned long long tag = (h >> 40) | 0x800000ULL;            // never zero
    unsigned long long slot = h & T.mask;
    for (unsigned long long probes = 0; probes <= T.mask; ++probes, slot = (slot + 1) & T.mask) {
        unsigned long long k = ld_cg64(&T.slots[slot].key);
        if (k == 0) {
            if (my_off < 0) {
                unsigned long long words = 1 + ((unsigned long long)len + 7) / 8;
                unsigned long long off = atomic_add64_warp(&T.cursor[0], words);
                if (off + words > T.arena_words) { atomic_or(T.err, AMP_E_ARENA_FULL); return; }
                unsigned char* rec = T.arena + off * 8;
                ((int*)rec)[0] = gpos; ((unsigned int*)rec)[1] = (unsigned int)len;
                for (int i = 0; i < len; i += 4) ((unsigned int*)(rec + 8))[i >> 2] = text.word(i, len);   // records are padded to 8 bytes
                fence();
                my_off = (long long)off;
            }
            unsigned long long old = atomic_cas64(&T.slots[slot].key, 0ULL, (tag << 40) | (unsigned long long)my_off);
            if (old == 0) {
                atomic_add(&T.slots[slot].count, n);
                const unsigned long long k_new = atomic_add64_warp(&T.cursor[1], 1ULL);
                T.entries[k_new] = (unsigned int)slot; T.slot_entry[slot] = (int)k_new;
                // the allele joins its position's list here, where it is created, so the lists are current after every
                // launch that adds alleles; their order is that of the exchanges (calling does not depend on it)
                if (T.heads) T.slots[slot].next = atomic_exch(&T.heads[gpos], (int)slot);
                return;
            }
            k = old;
        }
        if ((k >> 40) == tag && ins_rec_equal(T, k, gpos, len, text)) { atomic_add(&T.slots[slot].count, n); return; }
    }
    atomic_or(T.err, AMP_E_TABLE_FULL);
}
// The slot of an allele that is already in the table, -1 if it is not: the same hash and comparison as ins_table_add, nothing
// is written.
template <class Text>
AMP_HD int ins_table_find(const InsTable& T, int gpos, int len, const Text& text) {
    unsigned long long h = ins_hash_init(gpos);
    for (int i = 0; i < len; i += 4) h = ins_hash_word(h, text.word(i, len));
    h = ins_hash_final(h, len);
    const unsigned long long tag = (h >> 40) | 0x800000ULL;
    unsigned long long slot = h & T.mask;
    for (unsigned long long probes = 0; probes <= T.mask; ++probes, slot = (slot + 1) & T.mask) {
        const unsigned long long k = ld_cg64(&T.slots[slot].key);
        if (k == 0) return -1;
        if ((k >> 40) == tag && ins_rec_equal(T, k, gpos, len, text)) return (int)slot;
    }
    return -1;
}

// ---- pileup plan: walk the (trimmed) CIGAR exactly as update_base_counts walks get_aligned_pairs() ----
// Sink interface:  match(rpos, q, len)   aligned run (quality filter applied when counting)
//                  del(rpos, len, qa)    D / N run -> '-' channel, unconditional (714-715); qa = query index of the anchor
//                                        base of a D directly after M / = / X (the op's last base), -1 otherwise (N too)
//                  ins(pos, s_begin, s_len, q0)   insertion allele = query_seq[s_begin : s_begin + s_len]; q0 = the first
//                                        inserted base that passed the gates 718 / 722 (s_begin == q0: the key of 735-736)
// Returns AMP_E_* bits (0 = ok).
template <class Sink>
AMP_HD int plan_read(const uint32_t* c, int nc, int pos, int l_seq, const uint8_t* qual, int minq, int L, Sink& sink) {
    const int qs = q_align_start(c, nc);                      // 700
    const int qe = q_align_end(c, nc, l_seq);                 // 701
    const int ref_end = pos + ref_len_of(c, nc);              // 705
    // Errors are raised where the reference would raise them: a reference position outside the genome when it is indexed
    // (a fully clipped read at pos == L indexes nothing), a query index past l_seq when its quality is looked up (a CIGAR
    // whose P ops overrun the read still finishes through the break at 726 when the trailing clip comes first).
    if (pos < 0) return AMP_E_COORD;
    for (int k = 0; k < nc; ++k) if (c_op(c[k]) > OP_X) return AMP_E_CIGAR;
    int q = 0, r = pos, q0 = -1;   // q0 >= 0: an insertion event is open (730-734)
    bool after_m = false;          // the previous op walked (H and empty ops are skipped) was M / = / X
    // key slice [q0-1 : end) with python's negative-index wrap for q0 == 0
#define AMP_KEY(end_, at_) do { int b_ = q0 - 1; if (b_ < 0) { b_ += l_seq; if (b_ < 0) b_ = 0; } \
        int e_ = (end_) < l_seq ? (end_) : l_seq; int n_ = e_ - b_; if (n_ < 0) n_ = 0; \
        int p_ = (at_) - 1; if (p_ < 0) p_ = 0; if (p_ >= L) return AMP_E_COORD; sink.ins(p_, b_, n_, q0); q0 = -1; } while (0)
    for (int k = 0; k < nc; ++k) {
        const uint32_t op = c_op(c[k]); const int n = c_len(c[k]);
        if (op == OP_H || n == 0) continue;
        if (cons_qr(op)) {
            if (r + n > L) return AMP_E_COORD;
            if (q + n > l_seq) return AMP_E_CIGAR;
            if (q0 >= 0) {                                    // exit (A)/(A'): next pair is a match
                if (r == 0) { int e_ = q + 1 < l_seq ? q + 1 : l_seq; sink.ins(0, q0, e_ - q0, q0); q0 = -1; }   // 735-736
                else AMP_KEY(q, r);
            }
            sink.match(r, q, n);
            q += n; r += n;
            after_m = true;
            continue;
        } else if (op == OP_D || op == OP_N) {
            if (r + n > L) return AMP_E_COORD;
            if (q0 >= 0) {                                    // exit (B): key runs to the end of the read
                if (r == 0) return AMP_E_INS_END;             // None + 1 -> TypeError in the reference
                AMP_KEY(l_seq, r);
            }
            sink.del(r, n, op == OP_D && after_m ? q - 1 : -1);
            r += n;
        } else {                                              // I, S, P: pairs (q, None)
            int j = q; const int hi = q + n;
            if (q0 < 0 && j < qs) j = hi < qs ? hi : qs;      // rules 718/722 both skip: leading clip
            for (; j < hi; ++j) {
                if (q0 < 0 && j >= qe) return 0;   // trailing clip: every later pair is skipped (718) or breaks (726)
                if (j >= l_seq) return AMP_E_CIGAR;           // quality lookup past the read (IndexError, 718)
                if (q0 >= 0) {
                    if (j >= qe) { AMP_KEY(j, ref_end); }                  // exit (C), pair consumed
                    else if (qual[j] < minq) { AMP_KEY(j, ref_end); }      // exit (D), pair consumed
                } else {
                    if (qual[j] < minq) continue;                          // 718
                    if (j < qs) continue;                                  // 722
                    if (j >= qe) return 0;                                 // 726: break
                    q0 = j;                                                // 732
                }
            }
            q += n;
        }
        after_m = false;
    }
#undef AMP_KEY
    if (q0 >= 0) return AMP_E_INS_END;                        // IndexError at 734
    return 0;
}

// A unit of counting work produced by plan_read: an aligned run or a deletion run.
struct Seg {
    int rpos;            // first reference position
    int len;             // bases (30 bits); bit 31 = deletion run; bit 30 = offsets below are staging-buffer relative
    uint32_t qabs;       // index of the first base's quality (staging buffer or batch qual array)
    uint32_t nibabs;     // nibble index of the first base (staging buffer or batch seq array)
};

}  // namespace amp
