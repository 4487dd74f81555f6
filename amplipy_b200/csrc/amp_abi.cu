// amp_abi.cu -- kernels' __global__ wrappers + the C ABI declared in include/amplipy_b200.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/amplipy_b200.h"
#include "amp_warp.cuh"
#include "amp_call.cuh"
#include "amp_bgzf.cuh"
#include "amp_ont.cuh"
#include "amp_deflate.cuh"
#include "amp_ivar.cuh"
#include "amp_contig.cuh"
#include "amp_annot.cuh"
#include "amp_exchange.cuh"

static_assert(AMP_F_TRIM_START == AMP_FLAG_TRIM_START && AMP_F_KEEP == AMP_FLAG_KEEP && AMP_F_SKIPPED == AMP_FLAG_SKIPPED &&
                  AMP_F_ERROR == AMP_FLAG_ERROR && AMP_E_ARENA_FULL == AMP_DEVERR_ARENA_FULL &&
                  AMP_E_QSTATS_MISS == AMP_DEVERR_QSTATS_MISS && AMP_E_DELS_FULL == AMP_DEVERR_DELS_FULL,
              "flag constants out of sync with include/amplipy_b200.h");
static_assert(sizeof(amp::Seg) == 16 && sizeof(amp::InsSlot) == 16 && sizeof(amp::DelSlot) == 24, "layout");

namespace {

thread_local std::string g_err;
int fail(int code, const char* what, const char* detail = "") {
    g_err = std::string(what) + (detail[0] ? ": " : "") + detail;
    return code;
}
#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            char buf_[256];                                                                       \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
            g_err = buf_;                                                                         \
            return AMP_ERR_CUDA;                                                                  \
        }                                                                                         \
    } while (0)

#ifndef AMP_THREADS
#define AMP_THREADS 256
#endif
constexpr int kThreads = AMP_THREADS;
#ifndef AMP_CTAS
#define AMP_CTAS 4
#endif
constexpr int kCtasPerSm = AMP_CTAS;

// ---------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------
// two variants of the fused kernel: short-read batches (runs are counted warp-per-run) and indel-rich batches
// (generic-path reads count their own runs); see amp::cta_trim_pileup
__global__ void __launch_bounds__(kThreads, kCtasPerSm) amp_trim_pileup_kernel(const __grid_constant__ amp::KParams P) {
    extern __shared__ __align__(16) unsigned char smem[];
    amp::cta_trim_pileup<false>(P, smem, (int)blockIdx.x, (int)blockDim.x);
}
__global__ void __launch_bounds__(kThreads, kCtasPerSm) amp_trim_pileup_indel_kernel(const __grid_constant__ amp::KParams P) {
    extern __shared__ __align__(16) unsigned char smem[];
    amp::cta_trim_pileup<true>(P, smem, (int)blockIdx.x, (int)blockDim.x);
}

// warp-autonomous kernel for short-read batches (amp_warp.cuh): one CTA per SM, AMP7_WARPS independent warps
template <bool TRIM, bool PILE>
__global__ void __launch_bounds__(AMP7_WARPS * 32, 1) amp_trim_pileup_warp_kernel(const __grid_constant__ amp::KParams P) {
    extern __shared__ __align__(128) unsigned char smem7[];
    amp::cta_trim_pileup_v9<TRIM, PILE, AMP7_WT>(P, smem7, AMP7_GWARPS, AMP7_DWARPS);
}

// warp-per-read kernel for indel-rich batches (amp_ont.cuh): one CTA per SM, AMPO_WARPS warps
template <bool TRIM, bool PILE>
__global__ void __launch_bounds__(AMPO_WARPS * 32, 1) amp_trim_pileup_ont_kernel(const __grid_constant__ amp::KParams P) {
    extern __shared__ __align__(128) unsigned char smem_o[];
    amp::cta_trim_pileup_ont<TRIM, PILE, AMPO_WT>(P, smem_o, AMPO_GWARPS);
}

__device__ const unsigned char kFixedSyms[8] = {'A', 'C', 'G', 'T', 'N', '-', 0, 0};

// Calling (amp_call.cuh): sixteen lanes per (sample, position)
__global__ void __launch_bounds__(256) amp_call_kernel(const __grid_constant__ amp::CallParams P) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t / AMP_CALL_LANES >= (long long)P.n_samples * P.L) return;   // whole groups: blockDim is a multiple of 16
    amp::call_thread(P, kFixedSyms, t, (int)(threadIdx.x & 31));
}

// Strand / quality pass (amp_ivar.cuh): one CTA per AMP_QS_READS reads, after the fused kernel on the same stream
__global__ void __launch_bounds__(AMP_QS_READS) amp_qstats_kernel(const __grid_constant__ amp::QStatsParams P) {
    __shared__ int trev[AMP_NCH * AMP_QS_WT], tq[AMP_NCH * AMP_QS_WT];
    __shared__ int lo;
    amp::cta_qstats(P, trev, tq, &lo, (int)blockIdx.x, (int)blockDim.x);
}

// The same pass on a context with the deletion-allele table (amp_dels_enable): the anchored deletion events go to the table too
__global__ void __launch_bounds__(AMP_QS_READS) amp_qstats_dels_kernel(const __grid_constant__ amp::QStatsParams P) {
    __shared__ int trev[AMP_NCH * AMP_QS_WT], tq[AMP_NCH * AMP_QS_WT];
    __shared__ int lo;
    amp::cta_qstats<true>(P, trev, tq, &lo, (int)blockIdx.x, (int)blockDim.x);
}

// iVar calling (amp_ivar.cuh): one thread per (sample, position), after amp_call_kernel on its outputs
__global__ void __launch_bounds__(256) amp_ivar_kernel(const __grid_constant__ amp::IvarParams P) {
    const long long gp = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (gp < (long long)P.n_samples * P.L) amp::ivar_position(P, gp);
}

// iVar calling of the deletion alleles (amp_ivar.cuh): one thread per listed allele
__global__ void __launch_bounds__(256) amp_ivar_dels_kernel(const __grid_constant__ amp::IvarDelParams P) {
    const unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (k < P.n) amp::ivar_del(P, k);
}

// the deletion alleles in list order: key, count | rev << 32, qsum
__global__ void amp_dels_gather_kernel(amp::DelTable T, unsigned long long n, unsigned long long* o) {
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x) {
        const amp::DelSlot s = T.slots[T.entries[k]];
        o[3 * k] = s.key; o[3 * k + 1] = s.cr; o[3 * k + 2] = s.qsum;
    }
}

// alleles given as {key, count | rev << 32, qsum} added to the table (amp_dels_merge)
__global__ void amp_dels_merge_kernel(amp::DelTable T, unsigned long long n, const unsigned long long* in) {
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x)
        amp::del_table_add(T, (int)(in[3 * k] >> 32), (int)(in[3 * k] & 0xFFFFFFFFu), (unsigned int)in[3 * k + 1],
                           (unsigned int)(in[3 * k + 1] >> 32), in[3 * k + 2]);
}

// Reset of the deletion table, one block: its listed slots, then its cursor.  Runs on the stream of amp_reset_kernel, which
// clears the error word.
__global__ void __launch_bounds__(1024) amp_dels_reset_kernel(amp::DelTable T) {
    const unsigned long long n = T.cursor[0];
    for (unsigned long long k = threadIdx.x; k < n; k += blockDim.x) {
        amp::DelSlot z; z.key = 0; z.cr = 0; z.qsum = 0;
        T.slots[T.entries[k]] = z;
    }
    __syncthreads();
    if (threadIdx.x == 0) T.cursor[0] = 0;
}

// the per-slot stats of the insertion alleles in amp_ins_export order
__global__ void amp_qstats_gather_kernel(const unsigned int* entries, unsigned long long n, const int* ins_rev, const unsigned long long* ins_qsum,
                                         const unsigned char* ins_head, int* o_rev, unsigned long long* o_qsum, unsigned char* o_head) {
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned int s = entries[k];
        o_rev[k] = ins_rev[s]; o_qsum[k] = ins_qsum[s]; o_head[k] = ins_head[s];
    }
}

// Reset between samples, one launch: the count matrix (zero) and the list heads (-1) with 16-byte stores, the slots
// listed in entries[0, cursor[1]) -- the table was zero after amp_create / amp_reset and every slot taken since then is
// listed there, so clearing those is enough (the full table is tens of MB) -- and, by the last block to finish, the two
// cursors, the error word and the block counter itself.  Every block reads cursor[1] before it is counted as done.
// STATS: the strand / quality sums are enabled; their per-position sums and the listed slots' sums are zeroed too.
template <bool STATS>
__global__ void __launch_bounds__(256) amp_reset_kernel(uint4* counts, unsigned long long counts16, uint4* heads, unsigned long long heads16,
                                                        amp::InsSlot* slots, const unsigned int* entries, unsigned long long* cursor,
                                                        unsigned int* err, unsigned int* done, uint4* rev, uint4* qsum, unsigned long long stats16,
                                                        int* ins_rev, unsigned long long* ins_qsum, unsigned char* ins_head) {
    const unsigned long long n = cursor[1];
    const unsigned long long tid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long k = tid; k < counts16; k += nth) counts[k] = make_uint4(0u, 0u, 0u, 0u);
    for (unsigned long long k = tid; k < heads16; k += nth) heads[k] = make_uint4(~0u, ~0u, ~0u, ~0u);
    if (STATS)
        for (unsigned long long k = tid; k < stats16; k += nth) { rev[k] = make_uint4(0u, 0u, 0u, 0u); qsum[2 * k] = qsum[2 * k + 1] = make_uint4(0u, 0u, 0u, 0u); }
    for (unsigned long long k = tid; k < n; k += nth) {
        amp::InsSlot z; z.key = 0; z.count = 0; z.next = 0;
        slots[entries[k]] = z;
        if (STATS) { ins_rev[entries[k]] = 0; ins_qsum[entries[k]] = 0; ins_head[entries[k]] = 0; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(done, 1u) == gridDim.x - 1) { cursor[0] = 0; cursor[1] = 0; *err = 0; *done = 0; }
    }
}

__global__ void amp_gather_entries_kernel(const amp::InsSlot* slots, const unsigned int* entries, unsigned long long n,
                                          int* count, unsigned long long* off) {
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const amp::InsSlot s = slots[entries[k]];
        count[k] = s.count;
        off[k] = s.key & 0xFFFFFFFFFFULL;
    }
}

struct RawText {
    const char* p;
    __device__ char operator()(int i) const { return p[i]; }
    __device__ uint32_t word(int i, int len) const {
        uint32_t w = 0;
        for (int j = 0; j < 4 && i + j < len; ++j) w |= (uint32_t)(unsigned char)p[i + j] << (8 * j);
        return w;
    }
};
__global__ void amp_merge_kernel(amp::InsTable tab, long long n, const int* gpos, const int* count, const long long* str_off,
                                 const char* chars) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        RawText t{chars + str_off[k]};
        amp::ins_table_add(tab, gpos[k], (int)(str_off[k + 1] - str_off[k]), t, count[k]);
    }
}

// ---- deep-sample exchange (SURVEY.md 8e): a rank's insertion table packed into one fixed-size slot, all slots gathered
// with one collective, everybody else's alleles merged by one kernel -- no host round trip, no size negotiation.
// slot = { u64 n_alleles, u64 arena_words, {u64 arena word offset, u64 count}[cap_entries], arena bytes [cap_arena] }
__global__ void amp_ins_pack_kernel(amp::InsTable tab, unsigned long long* slot, unsigned long long cap_entries,
                                    unsigned long long cap_arena_words) {
    // cursor[0] runs past the arena when a reservation failed (AMP_E_ARENA_FULL); no slot names such a record
    const unsigned long long words = tab.cursor[0] < tab.arena_words ? tab.cursor[0] : tab.arena_words, n = tab.cursor[1];
    const bool fits = n <= cap_entries && words <= cap_arena_words;
    const unsigned long long tid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
    if (tid == 0) {
        slot[0] = fits ? n : 0ULL; slot[1] = fits ? words : 0ULL;
        if (!fits) atomicOr(tab.err, n > cap_entries ? AMP_E_TABLE_FULL : AMP_E_ARENA_FULL);
    }
    if (!fits) return;
    unsigned long long* ent = slot + 2;
    for (unsigned long long k = tid; k < n; k += nth) {
        const amp::InsSlot s = tab.slots[tab.entries[k]];
        ent[2 * k] = s.key & 0xFFFFFFFFFFULL; ent[2 * k + 1] = (unsigned long long)(unsigned int)s.count;
    }
    unsigned long long* dst = slot + 2 + 2 * cap_entries;
    const unsigned long long* src = (const unsigned long long*)tab.arena;
    for (unsigned long long k = tid; k < words; k += nth) dst[k] = src[k];
}
__global__ void amp_ins_merge_packed_kernel(amp::InsTable tab, const unsigned long long* slots, unsigned long long slot_words,
                                            unsigned long long cap_entries, int my_rank) {
    const int r = (int)blockIdx.y;
    if (r == my_rank) return;
    const unsigned long long* slot = slots + (unsigned long long)r * slot_words;
    const unsigned long long n = slot[0];
    const unsigned long long* ent = slot + 2;
    const unsigned char* arena = (const unsigned char*)(slot + 2 + 2 * cap_entries);
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned char* rec = arena + ent[2 * k] * 8;
        const int gpos = ((const int*)rec)[0];
        const int len = (int)((const unsigned int*)rec)[1];
        amp::ArenaText t{rec + 8};
        amp::ins_table_add(tab, gpos, len, t, (int)ent[2 * k + 1]);
    }
}

// The same two steps for a context with the strand / quality sums (amp_exchange.cuh): every entry carries its allele's sums.
__global__ void amp_ins_pack_qstats_kernel(amp::InsTable tab, amp::QStatsSlots q, unsigned long long* slot, unsigned long long cap_entries,
                                           unsigned long long cap_arena_words) {
    unsigned long long n, words;
    const bool fits = amp::xq_pack_size(tab, cap_entries, cap_arena_words, n, words);
    const unsigned long long tid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
    if (tid == 0) amp::xq_pack_header(tab, slot, fits, n, words, cap_entries);
    if (!fits) return;
    for (unsigned long long k = tid; k < n; k += nth) amp::xq_pack_entry(tab, q, slot, k);
    unsigned long long* dst = amp::xq_slot_arena(slot, cap_entries);
    const unsigned long long* src = (const unsigned long long*)tab.arena;
    for (unsigned long long k = tid; k < words; k += nth) dst[k] = src[k];
}
__global__ void amp_ins_merge_packed_qstats_kernel(amp::InsTable tab, amp::QStatsSlots q, const unsigned long long* slots,
                                                   unsigned long long slot_words, unsigned long long cap_entries, int my_rank) {
    const int r = (int)blockIdx.y;
    if (r == my_rank) return;
    const unsigned long long* slot = slots + (unsigned long long)r * slot_words;
    const unsigned long long n = slot[0];
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x)
        amp::xq_merge_entry(tab, q, slot, cap_entries, k);
}

// The deletion table of a rank packed into one fixed-size slot and the other ranks' slots merged (amp_exchange.cuh)
__global__ void amp_dels_pack_kernel(amp::DelTable T, unsigned long long* slot, unsigned long long cap_entries) {
    unsigned long long n;
    const bool fits = amp::xd_pack_size(T, cap_entries, n);
    const unsigned long long tid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
    if (tid == 0) amp::xd_pack_header(T, slot, fits, n);
    if (!fits) return;
    for (unsigned long long k = tid; k < n; k += nth) amp::xd_pack_entry(T, slot, k);
}
__global__ void amp_dels_merge_packed_kernel(amp::DelTable T, const unsigned long long* slots, unsigned long long slot_words, int my_rank) {
    const int r = (int)blockIdx.y;
    if (r == my_rank) return;
    const unsigned long long* slot = slots + (unsigned long long)r * slot_words;
    const unsigned long long n = slot[0];
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += (unsigned long long)gridDim.x * blockDim.x)
        amp::xd_merge_entry(T, slot, k);
}

// ---- BGZF deflate on the device (amp_deflate.cuh) --------------------------------------------------------------------------
#define AMPD_WARPS 24
// block k = in[bstart[k], bstart[k + 1]) -> a deflate stream in slot k (clen[k] = its bytes, 0xFFFFFFFF: did not shrink, to be stored)
// and its CRC-32; the warps take blocks from a counter
__global__ void __launch_bounds__(AMPD_WARPS * 32) amp_bgzf_deflate_kernel(const uint8_t* in, const long long* bstart, long long nb, uint8_t* slots,
                                                                          uint32_t* clen, uint32_t* crc, unsigned int* next, uint32_t* toks) {
    extern __shared__ __align__(16) unsigned char dsm[];
    amp::DeflateTables& T = *(amp::DeflateTables*)dsm;
    amp::DeflateMem& M = ((amp::DeflateMem*)(dsm + ((sizeof(amp::DeflateTables) + 15) & ~(size_t)15)))[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    amp::deflate_tables_init(T, (int)threadIdx.x, (int)blockDim.x);
    __syncthreads();
    const uint32_t mcol = amp::crc_shift_column(T, lane);
    for (;;) {
        unsigned int t = 0;
        if (lane == 0) t = atomicAdd(next, 1u);
        const long long k = (long long)__shfl_sync(0xFFFFFFFFu, t, 0);
        if (k >= nb) break;
        const uint8_t* src = in + bstart[k];
        const int n = (int)(bstart[k + 1] - bstart[k]);
        const int cap_words = (n + 3) / 4;                                // "does not shrink" = would need more words than the input has
        uint32_t* tok = toks + ((size_t)blockIdx.x * AMPD_WARPS + (threadIdx.x >> 5)) * AMPD_SCRATCH;
        int bytes = n >= 16 ? amp::deflate_block(src, n, M, T, (uint32_t*)(slots + (size_t)k * AMPD_SLOT), cap_words, tok, lane) : -1;
        if (bytes >= n + 5) bytes = -1;
        const uint32_t cr = amp::crc32_block(src, n, T, mcol, lane);
        if (lane == 0) { clen[k] = bytes < 0 ? 0xFFFFFFFFu : (uint32_t)bytes; crc[k] = cr; }
        __syncwarp();
    }
}
// the BGZF blocks themselves: 18-byte header, the deflate stream (or the data as one stored block), CRC-32, ISIZE, at off[k]
__global__ void __launch_bounds__(256) amp_bgzf_pack_kernel(const uint8_t* in, const long long* bstart, long long nb, const uint8_t* slots,
                                                           const uint32_t* clen, const uint32_t* crc, const long long* off, uint8_t* out) {
    const int lane = threadIdx.x & 31;
    const long long k = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= nb) return;
    const uint32_t n = (uint32_t)(bstart[k + 1] - bstart[k]);
    const bool stored = clen[k] == 0xFFFFFFFFu;
    const uint32_t payload = stored ? n + 5u : clen[k], bsize = payload + 26u;
    uint8_t* dst = out + off[k];
    if (lane < 18) {
        const uint8_t hdr[18] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, (uint8_t)((bsize - 1u) & 0xFFu), (uint8_t)((bsize - 1u) >> 8)};
        dst[lane] = hdr[lane];
    }
    uint8_t* pay = dst + 18;
    if (stored) {
        if (lane == 0) { pay[0] = 1; pay[1] = (uint8_t)(n & 0xFFu); pay[2] = (uint8_t)(n >> 8); pay[3] = (uint8_t)(~n & 0xFFu); pay[4] = (uint8_t)((~n >> 8) & 0xFFu); }
        const uint8_t* src = in + bstart[k];
        for (uint32_t i = lane; i < n; i += 32) pay[5 + i] = src[i];
    } else {
        const uint8_t* src = slots + (size_t)k * AMPD_SLOT;
        for (uint32_t i = lane; i < payload; i += 32) pay[i] = src[i];
    }
    if (lane < 8) { const uint32_t v = lane < 4 ? crc[k] : n; pay[payload + lane] = (uint8_t)(v >> (8 * (lane & 3))); }
}

// ---- trimmed BAM records rebuilt on the device (what assigning cigartuples / reference_start does to a pysam segment before
// out_aln.write, AmpliPy.py:463-514, 591-658, 911): everything but pos / bin / n_cigar / CIGAR is copied byte for byte ------------------
// size of read i's record in the output (0: the read does not pass the write gate, AmpliPy.py:910)
__global__ void amp_bam_newsize_kernel(const uint8_t* raw, const unsigned long long* rec_off, long long n, const uint16_t* o_ncig, const uint8_t* o_flags,
                                       uint32_t* sizes) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sizes[i] = (o_flags[i] & AMP_F_KEEP) ? amp::bam_new_record_size(raw, rec_off[i], (uint32_t)o_ncig[i]) : 0u;
}
// exclusive prefix sums of n 32-bit sizes (64-bit results, n + 1 of them), one CTA
__global__ void __launch_bounds__(1024) amp_scan_sizes_kernel(const uint32_t* sizes, long long n, unsigned long long* off) {
    __shared__ unsigned long long part[1024];
    const int t = threadIdx.x;
    const long long per = (n + 1023) / 1024, lo = t * per, hi = lo + per < n ? lo + per : n;
    unsigned long long s = 0;
    for (long long k = lo; k < hi; ++k) s += sizes[k];
    part[t] = s;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const unsigned long long v = t >= d ? part[t - d] : 0ULL;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    unsigned long long run = part[t] - s;
    for (long long k = lo; k < hi; ++k) { off[k] = run; run += sizes[k]; }
    if (t == 1023) off[n] = part[1023];
}
// one warp per kept read: the record with its new block_size / pos / bin / n_cigar / CIGAR at out + off[i]
__global__ void __launch_bounds__(256) amp_bam_rewrite_kernel(const uint8_t* raw, const unsigned long long* rec_off, long long n, const uint32_t* cig_off,
                                                             const int32_t* o_pos, const uint16_t* o_ncig, const uint32_t* o_cigar,
                                                             const unsigned long long* off, uint8_t* out) {
    const int lane = threadIdx.x & 31;
    const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n || off[i + 1] == off[i]) return;
    amp::bam_rewrite_record(raw, rec_off[i], o_pos[i], o_cigar + (size_t)cig_off[i] + 3 * (size_t)i, (uint32_t)o_ncig[i], out + off[i], lane);
}

// ---- BGZF / BAM decode on the device (amp_bgzf.cuh) ------------------------------------------------------------------------
#define AMPZ_WARPS 16
__global__ void __launch_bounds__(AMPZ_WARPS * 32) amp_bgzf_inflate_kernel(const uint8_t* comp, long long comp_len, const long long* in_off,
                                                                          const uint32_t* out_len, const long long* out_off, long long k0,
                                                                          long long k1, uint8_t* raw, unsigned int* next, unsigned int* err) {
    extern __shared__ __align__(16) unsigned char zsm[];
    amp::InflateMem& M = ((amp::InflateMem*)zsm)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    for (;;) {
        unsigned int t = 0;
        if (lane == 0) t = atomicAdd(next, 1u);
        const long long k = k0 + (long long)__shfl_sync(0xFFFFFFFFu, t, 0);
        if (k >= k1) break;
        const uint8_t* b = comp + in_off[k];
        const long long bend = in_off[k + 1];                 // (the table has one entry more: the end of the last block)
        const long long xlen = (long long)b[10] | ((long long)b[11] << 8);
        const long long clen = bend - in_off[k] - 12 - xlen - 8;
        int e = 0;
        if (clen < 0) e = AMPZ_E_DATA;
        else if (out_len[k]) e = amp::inflate_block(b + 12 + xlen, clen, raw + out_off[k], (long long)out_len[k], M, lane);
        if (e && lane == 0) atomicOr(err, (unsigned int)e);
        __syncwarp();
    }
}
__global__ void amp_bam_count_kernel(const uint8_t* raw, const long long* out_off, long long n_blocks, long long body_off,
                                     amp::BamBlockTotals* tot, unsigned int* err) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n_blocks) return;
    long long lo = out_off[k]; const long long hi = out_off[k + 1];
    if (lo < body_off) lo = body_off;
    amp::BamBlockTotals t; t.n_rec = 0; t.n_cig = 0; t.n_seq = 0; t.n_qual = 0;
    if (lo < hi && !amp::bam_chain_totals(raw, lo, hi, t)) { atomicOr(err, (unsigned int)AMPZ_E_ALIGN); t.n_rec = 0; t.n_cig = 0; t.n_seq = 0; t.n_qual = 0; }
    tot[k] = t;
}
// exclusive prefix sums of the per-block totals (one CTA): prefix[c][k], c = records, CIGAR ops, seq bytes, qual bytes; prefix[c][n] = total
__global__ void __launch_bounds__(1024) amp_bam_scan_kernel(const amp::BamBlockTotals* tot, long long n_blocks, unsigned long long* prefix) {
    __shared__ unsigned long long part[4][1024];
    const int t = threadIdx.x;
    const long long per = (n_blocks + 1023) / 1024, lo = t * per, hi = lo + per < n_blocks ? lo + per : n_blocks;
    unsigned long long s[4] = {0, 0, 0, 0};
    for (long long k = lo; k < hi; ++k) { s[0] += tot[k].n_rec; s[1] += tot[k].n_cig; s[2] += tot[k].n_seq; s[3] += tot[k].n_qual; }
    for (int c = 0; c < 4; ++c) part[c][t] = s[c];
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        unsigned long long v[4];
        for (int c = 0; c < 4; ++c) v[c] = t >= d ? part[c][t - d] : 0ULL;
        __syncthreads();
        for (int c = 0; c < 4; ++c) part[c][t] += v[c];
        __syncthreads();
    }
    unsigned long long run[4];
    for (int c = 0; c < 4; ++c) run[c] = part[c][t] - s[c];
    for (long long k = lo; k < hi; ++k) {
        for (int c = 0; c < 4; ++c) prefix[(size_t)c * (n_blocks + 1) + k] = run[c];
        run[0] += tot[k].n_rec; run[1] += tot[k].n_cig; run[2] += tot[k].n_seq; run[3] += tot[k].n_qual;
    }
    if (t == 1023) for (int c = 0; c < 4; ++c) prefix[(size_t)c * (n_blocks + 1) + n_blocks] = part[c][1023];
}
__global__ void __launch_bounds__(256) amp_bam_scatter_kernel(const uint8_t* raw, const long long* out_off, long long n_blocks, long long body_off,
                                                             const unsigned long long* prefix, amp::BamSoa D) {
    const long long k = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= n_blocks) return;
    long long lo = out_off[k]; const long long hi = out_off[k + 1];
    if (lo < body_off) lo = body_off;
    const size_t st = (size_t)(n_blocks + 1);
    if (lo < hi) amp::bam_scatter_block(raw, lo, hi, D, prefix[k], prefix[st + k], prefix[2 * st + k], prefix[3 * st + k], lane);
    if (k == n_blocks - 1 && lane == 0) {                     // the closing entries of the three offset arrays
        const unsigned long long n = prefix[n_blocks];
        D.cig_off[n] = (uint32_t)prefix[st + n_blocks]; D.seq_off[n] = (uint32_t)prefix[2 * st + n_blocks]; D.qual_off[n] = (uint32_t)prefix[3 * st + n_blocks];
    }
}

// ---- a batch grouped by contig (amp_contig.cuh): plan, stable counting sort, permuted copy, outputs back to input order ----------
__global__ void __launch_bounds__(AMP_CT_THREADS) amp_contig_plan_kernel(const __grid_constant__ amp::ContigPlanParams P) {
    __shared__ amp::ContigPlanSmem sm;
    amp::contig_plan_cta(P, sm, (int)blockIdx.x);
}
__global__ void __launch_bounds__(AMP_CT_THREADS) amp_contig_scan_kernel(const __grid_constant__ amp::ContigScanParams P0,
                                                                        const __grid_constant__ amp::ContigScanParams P1,
                                                                        const __grid_constant__ amp::ContigScanParams P2) {
    __shared__ unsigned long long part[AMP_CT_THREADS];
    amp::contig_scan_cta(blockIdx.y == 0 ? P0 : blockIdx.y == 1 ? P1 : P2, part);
}
__global__ void __launch_bounds__(AMP_CT_THREADS) amp_contig_rank_kernel(const __grid_constant__ amp::ContigRankParams P) {
    __shared__ amp::ContigRankSmem sm;
    amp::contig_rank_cta(P, sm, (int)blockIdx.x);
}
__global__ void __launch_bounds__(AMP_CT_THREADS) amp_contig_tilesum_kernel(const __grid_constant__ amp::ContigGatherParams P) {
    __shared__ unsigned long long part[AMP_CT_THREADS];
    amp::contig_tilesum_cta(P, part, (int)blockIdx.x);
}
__global__ void __launch_bounds__(AMP_CT_THREADS) amp_contig_gather_kernel(const __grid_constant__ amp::ContigGatherParams P) {
    __shared__ unsigned long long part[AMP_CT_THREADS];
    amp::contig_gather_cta(P, part, (int)blockIdx.x);
}
__global__ void __launch_bounds__(256) amp_contig_unpermute_kernel(const __grid_constant__ amp::ContigUnpermuteParams P) {
    amp::contig_unpermute_warp(P, (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, ((long long)gridDim.x * blockDim.x) >> 5);
}
__global__ void __launch_bounds__(256) amp_contig_skip_kernel(const __grid_constant__ amp::ContigSkipParams P) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P.n; i += (long long)gridDim.x * blockDim.x) amp::contig_skip_read(P, i);
}

// ---- codon annotation (amp_annot.cuh): counts and per-tile sums, a scan of the tile sums (amp_contig_scan_kernel), then the
// offsets and the entries ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(AMP_AN_THREADS) amp_annot_count_kernel(const __grid_constant__ amp::AnnotParams P, uint32_t* tsum) {
    __shared__ unsigned int s;
    if (threadIdx.x == 0) s = 0;
    __syncthreads();
    const long long gp = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (gp < (long long)P.n_samples * P.L) {
        const unsigned int n = amp::annot_count(P, gp);
        P.off[gp] = n;
        if (n) atomicAdd(&s, n);
    }
    __syncthreads();
    if (threadIdx.x == 0) tsum[blockIdx.x] = s;
}
__global__ void __launch_bounds__(AMP_AN_THREADS) amp_annot_fill_kernel(const __grid_constant__ amp::AnnotParams P, const uint32_t* tbase,
                                                                        unsigned int n_tiles) {
    __shared__ unsigned long long part[AMP_AN_THREADS];
    const long long SL = (long long)P.n_samples * P.L;
    const long long gp = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const unsigned int n = gp < SL ? P.off[gp] : 0u;
    unsigned long long total;
    const unsigned int o = tbase[blockIdx.x] + (unsigned int)amp::cta_excl_scan(n, part, &total);
    if (gp < SL) {
        P.off[gp] = o;
        if (n) amp::annot_fill(P, gp, o);
    }
    if (gp == 0) P.off[SL] = tbase[n_tiles];
}

struct DevChunk {   // device staging for one in-flight chunk of amp_process_host
    cudaStream_t stream = nullptr;
    int32_t* pos = nullptr; uint16_t* flag = nullptr; int32_t* tlen = nullptr;
    uint32_t *cig_off = nullptr, *seq_off = nullptr, *qual_off = nullptr, *cigar = nullptr;
    uint8_t *seq = nullptr, *qual = nullptr;
    int32_t* o_pos = nullptr; uint16_t* o_ncig = nullptr; uint8_t* o_flags = nullptr; uint32_t* o_cigar = nullptr;
    uint32_t* scratch = nullptr;
    uint32_t* glist = nullptr; size_t cap_glist = 0;
    size_t cap_ocigar = 0;
    size_t cap_reads = 0, cap_cig = 0, cap_seq = 0, cap_qual = 0, cap_scratch = 0;
};

}  // namespace

struct amp_ctx {
    amp_config cfg;
    int Lpad = 0, sm_count = 0, max_primer_len = 0;
    int32_t *d_min_start = nullptr, *d_max_end = nullptr;
    // samples with a primer scheme / reference of their own (amp_set_scheme / amp_set_sample_reference; SURVEY.md 8f-4)
    struct Scheme { int32_t* d_min = nullptr; int32_t* d_max = nullptr; int L = 0, mpl = 0; };
    std::vector<Scheme> scheme;
    bool ref_per_sample = false;
    int* d_counts = nullptr; bool counts_owned = true;
    amp::InsTable tab{};
    unsigned long long nslots = 0;
    unsigned int* d_err = nullptr;
    unsigned int* d_reset_done = nullptr;   // block counter of amp_reset_kernel
    uint32_t* d_scratch = nullptr; size_t scratch_words = 0;
    uint32_t* d_glist = nullptr; size_t glist_words = 0;   // per-CTA generic-read lists of the warp-autonomous kernels
    DevChunk chunk[3];
    int last_launches = 0;
    size_t max_dyn_smem = 0;
    bool v7_attr = false, ont_attr = false;
    // decoded file (amp_bam_decode_host): compressed bytes, inflated stream, block tables, struct-of-arrays batch, trim outputs
    struct Decoded {
        uint8_t* comp = nullptr; size_t cap_comp = 0;
        uint8_t* raw = nullptr; size_t cap_raw = 0;
        long long* in_off = nullptr; long long* out_off = nullptr; uint32_t* out_len = nullptr; amp::BamBlockTotals* tot = nullptr;
        unsigned long long* prefix = nullptr; size_t cap_blocks = 0;
        unsigned int* ctr = nullptr;                              // [0] block counter of the inflate kernel, [1] error bits
        int32_t* pos = nullptr; uint16_t* flag = nullptr; int32_t* tlen = nullptr; uint32_t *cig_off = nullptr, *seq_off = nullptr, *qual_off = nullptr;
        unsigned long long* rec_off = nullptr; int32_t* o_pos = nullptr; uint16_t* o_ncig = nullptr; uint8_t* o_flags = nullptr; size_t cap_reads = 0;
        uint32_t* cigar = nullptr; size_t cap_cig = 0; uint8_t* seq = nullptr; size_t cap_seq = 0; uint8_t* qual = nullptr; size_t cap_qual = 0;
        uint32_t* o_cigar = nullptr; size_t cap_ocig = 0; uint32_t* scratch = nullptr; size_t cap_scratch = 0;
        long long n_reads = 0, sum_cig = 0, sum_seq = 0, sum_qual = 0, n_blocks = 0, raw_len = 0;
        bool valid = false, z_attr = false, trimmed = false;             // trimmed: o_* hold the trim outputs of this batch
        uint32_t* w_sizes = nullptr; size_t cap_wsizes = 0; unsigned long long* w_off = nullptr; size_t cap_woff = 0; uint8_t* w_stream = nullptr; size_t cap_wstream = 0;
        cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
        cudaStream_t zs[4] = {nullptr, nullptr, nullptr, nullptr};   // streams of the inflate launches 1..3
    } dec;
    struct Deflater {                                            // amp_bgzf_deflate_host (grown at high-water marks)
        uint8_t* in = nullptr; size_t cap_in = 0; uint8_t* slots = nullptr; size_t cap_slots = 0; uint8_t* out = nullptr; size_t cap_out = 0;
        long long* bstart = nullptr; size_t cap_bstart = 0; long long* off = nullptr; size_t cap_off = 0;
        uint32_t* clen = nullptr; size_t cap_clen = 0; uint32_t* crc = nullptr; size_t cap_crc = 0; unsigned int* ctr = nullptr;
        uint32_t* toks = nullptr; size_t cap_toks = 0;           // token scratch of the deflate kernel's warps
        bool attr = false; cudaStream_t stream = nullptr;            // its own stream: a writer thread may call it while the context calls
    } defl;
    unsigned char* d_xbuf = nullptr; size_t xbuf_bytes = 0;   // scratch of amp_ins_export / amp_ins_merge (grown at high-water marks)
    unsigned char* d_ref = nullptr;     // reference characters (amp_set_reference)
    unsigned char* d_call = nullptr;    // calling outputs (one block, offsets below)
    size_t o_depth = 0, o_top = 0, o_topc = 0, o_fl = 0, o_refc = 0, o_ff = 0, o_fr = 0, o_alt = 0, o_if = 0, o_ir = 0, o_ia = 0;
    // strand / quality stats (amp_qstats_enable): [n_samples][6][Lpad] sums and per-slot sums of the insertion alleles
    int* d_rev = nullptr; unsigned long long* d_qsum = nullptr;
    int* d_ins_rev = nullptr; unsigned long long* d_ins_qsum = nullptr; unsigned char* d_ins_head = nullptr;
    unsigned char* d_ivar = nullptr;    // iVar calling outputs (one block, offsets below)
    size_t o_iu = 0, o_fmq = 0, o_fpv = 0, o_imq = 0, o_ipv = 0;
    // anchored deletion alleles (amp_dels_enable): the table, and the calling outputs (mq, then pval; grown at high-water marks)
    amp::DelTable dels{}; unsigned long long dels_nslots = 0;
    unsigned long long* d_dels_out = nullptr; size_t dels_out_words = 0;
    // a batch grouped by contig (amp_contig_plan_* / amp_process_contigs; buffers grown at high-water marks)
    struct Contigs {
        int source = 0;                                           // the planned batch: 0 none, 1 the decoded one, 2 a device batch
        amp::BatchPtrs b{}; long long sum_cig = 0; bool grouped = false;   // the planned batch, its CIGAR ops, its plan's verdict
        int* sid = nullptr; size_t cap_sid = 0; uint32_t* hist = nullptr; size_t cap_hist = 0; uint32_t* hist_off = nullptr; size_t cap_hoff = 0;
        unsigned long long* table = nullptr; size_t cap_table = 0; std::vector<unsigned long long> h_table;
        uint32_t* perm = nullptr; size_t cap_perm = 0; uint32_t* tsum = nullptr; size_t cap_tsum = 0; uint32_t* tbase = nullptr; size_t cap_tbase = 0;
        int32_t* pos = nullptr; size_t cap_pos = 0; uint16_t* flag = nullptr; size_t cap_flag = 0; int32_t* tlen = nullptr; size_t cap_tlen = 0;
        uint32_t* cig_off = nullptr; size_t cap_coff = 0; uint32_t* seq_off = nullptr; size_t cap_soff = 0; uint32_t* qual_off = nullptr; size_t cap_qoff = 0;
        uint32_t* cigar = nullptr; size_t cap_cig = 0; uint8_t* seq = nullptr; size_t cap_seq = 0; uint8_t* qual = nullptr; size_t cap_qual = 0;
        int32_t* o_pos = nullptr; size_t cap_opos = 0; uint16_t* o_ncig = nullptr; size_t cap_oncig = 0; uint8_t* o_flags = nullptr; size_t cap_oflags = 0;
        uint32_t* o_cigar = nullptr; size_t cap_ocig = 0; uint32_t* scratch = nullptr; size_t cap_scratch = 0;
    } ct;
    std::vector<int> ref_len_s;         // per-sample reference lengths (amp_set_sample_reference)
    // codon annotation (amp_set_features / amp_annotate; buffers grown at high-water marks)
    struct Annot {
        std::vector<amp::AnnotFeatures> feat; bool built = false; long long n = 0;
        int* tables = nullptr; size_t cap_tables = 0; uint32_t* off = nullptr; size_t cap_off = 0;
        uint32_t* tsum = nullptr; size_t cap_tsum = 0; uint32_t* tbase = nullptr; size_t cap_tbase = 0;
        int* e_int = nullptr; size_t cap_eint = 0; unsigned char* e_chr = nullptr; size_t cap_echr = 0;   // feat, pos_aa | off, codons, aas
    } an;
};

namespace {

template <class T>
int dev_grow(T** p, size_t* cap, size_t need) {
    if (need <= *cap) return AMP_OK;
    if (*p) CK(cudaFree(*p));
    *p = nullptr; *cap = 0;
    size_t n = need + need / 4 + 64;
    CK(cudaMalloc((void**)p, n * sizeof(T)));
    *cap = n;
    return AMP_OK;
}

bool has_scheme(const amp_ctx* c, int sample) {
    return c->d_min_start || (sample >= 0 && (size_t)sample < c->scheme.size() && c->scheme[sample].L > 0);
}

// words of the per-CTA generic-read lists + their counters for a launch over n reads
size_t glist_words_for(const amp_ctx* c, long long n) { return (size_t)n + 33 * ((size_t)c->sm_count + 1) + (size_t)c->sm_count + 64; }

int launch_fused(amp_ctx* c, const amp::BatchPtrs& b, long long sum_cig, long long max_cig, long long sum_qual, int mode,
                 int sample, const amp::TrimOut& o, uint32_t* scratch, uint32_t* glist, cudaStream_t st) {
    if (b.n <= 0) return AMP_OK;
    amp::KParams P{};
    P.b = b; P.o = o;
    P.tp.L = c->cfg.ref_len; P.tp.min_primer_start = c->d_min_start; P.tp.max_primer_end = c->d_max_end;
    P.tp.max_primer_len = c->max_primer_len;
    if ((size_t)sample < c->scheme.size() && c->scheme[sample].L > 0) {       // this sample's own scheme
        const auto& sc = c->scheme[sample];
        P.tp.L = sc.L; P.tp.min_primer_start = sc.d_min; P.tp.max_primer_end = sc.d_max; P.tp.max_primer_len = sc.mpl;
    } P.tp.min_quality = c->cfg.min_quality; P.tp.window = c->cfg.sliding_window;
    P.tp.min_length = c->cfg.min_length; P.tp.include_no_primer = c->cfg.include_no_primer;
    P.mode = mode & (AMP_MODE_TRIM | AMP_MODE_PILEUP);
    P.counts = c->d_counts + (size_t)sample * AMP_NCH * c->Lpad;
    P.Lpad = c->Lpad; P.gpos_base = sample * c->Lpad;
    P.tab = c->tab; P.err = c->d_err;
    P.scratch = scratch; P.scratch_half = sum_cig + 3 * b.n;
    (void)max_cig;
    const amp::TileCfg t = amp::pick_tile_cfg(b.n, sum_cig, sum_qual, mode);
    // short-read batches: warp-autonomous kernel.  AMP_KERNEL=tile forces the older CTA-phased kernel (A/B experiments).
    static const bool force_tile = [] { const char* e = getenv("AMP_KERNEL"); return e && !strcmp(e, "tile"); }();
    static const bool force_warp = [] { const char* e = getenv("AMP_KERNEL"); return e && !strcmp(e, "warp"); }();
    if (force_warp || (!t.direct && !force_tile && sum_qual <= 1000 * b.n)) {
        const amp::V7Cfg v = amp::pick_v7_cfg(b.n, sum_qual, c->sm_count);
        P.wt = v.wt; P.reads_per_tile = v.batch_reads;
        P.ntiles = (int)((b.n + v.batch_reads - 1) / v.batch_reads);
        int grid = std::max(1, std::min(P.ntiles, c->sm_count));
        P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
        grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
        const size_t smem = amp::smem_bytes_v9(P.wt, AMP7_WARPS, AMP7_GWARPS);
        if (!c->v7_attr) {
            CK(cudaFuncSetAttribute(amp_trim_pileup_warp_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(amp_trim_pileup_warp_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(amp_trim_pileup_warp_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            c->v7_attr = true;
        }
        // per-CTA lists of the reads that need the generic phase
        P.gcap = (long long)P.tiles_per_cta * P.reads_per_tile;
        P.glist = glist;
#ifdef AMP7_TIMING
        static long long* d_phase7 = nullptr;
        if (!d_phase7) CK(cudaMalloc((void**)&d_phase7, 400 * 8));
        CK(cudaMemsetAsync(d_phase7, 0, 400 * 8, st));
        { const long long big = 1LL << 60; CK(cudaMemcpyAsync(d_phase7 + 9, &big, 8, cudaMemcpyHostToDevice, st)); }
        P.phase_cycles = d_phase7;
        P.direct = getenv("AMP7_REVERSE") ? 1 : 0;
#endif
        const bool tr = mode & AMP_MODE_TRIM, pl = mode & AMP_MODE_PILEUP;
        if (tr && pl) amp_trim_pileup_warp_kernel<true, true><<<grid, AMP7_WARPS * 32, smem, st>>>(P);
        else if (tr) amp_trim_pileup_warp_kernel<true, false><<<grid, AMP7_WARPS * 32, smem, st>>>(P);
        else amp_trim_pileup_warp_kernel<false, true><<<grid, AMP7_WARPS * 32, smem, st>>>(P);
        CK(cudaGetLastError());
#ifdef AMP7_TIMING
        {
            CK(cudaStreamSynchronize(st));
            long long h[400];
            CK(cudaMemcpy(h, d_phase7, sizeof h, cudaMemcpyDeviceToHost));
            if (getenv("AMP7_DUMP_CTAS")) { for (int b = 0; b < grid && b < 160; ++b) fprintf(stderr, "%lld:%lld ", h[16 + b] / 1000, h[176 + b]); fprintf(stderr, "\n"); }
            const double wf = (double)grid * AMP7_WARPS;
            fprintf(stderr, "[cycles per warp] prologue %.0f  A %.0f  bulk-wait %.0f  window+trim %.0f  count %.0f  (barrier issue %.0f)  wait+generic %.0f\n",
                    h[0] / wf, h[1] / wf, h[2] / wf, h[3] / wf, h[4] / wf, h[5] / wf, h[6] / wf);
            fprintf(stderr, "[generic phase, cycles summed over its warp-rounds / 1000] load+copy %lld  trim_read %lld  outputs %lld  plan_read %lld\n", h[360] / 1000, h[361] / 1000, h[362] / 1000, h[363] / 1000);
            fprintf(stderr, "[cycles per CTA] mean %.0f  min %lld  max %lld   set-up %.0f  last barrier (per warp) %.0f  drain+flush %.0f\n", (double)h[8] / grid, h[9], h[10],
                    (double)h[11] / grid, h[12] / wf, (double)h[13] / grid);
            fprintf(stderr, "[runs counted outside the tile] %lld\n", h[14]);
        }
#endif
        c->last_launches += 1;
        return AMP_OK;
    }
    // indel-rich batches: the warp-per-read kernel.  AMP_KERNEL=tile forces the older CTA-phased kernel (A/B experiments).
    if (t.direct && !force_tile && b.n < (1LL << 31)) {
        P.wt = AMPO_WT; P.reads_per_tile = 1;
        P.ntiles = (int)b.n;
        int grid = std::max(1, std::min(P.ntiles, c->sm_count));
        P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
        grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
        const size_t smem = amp::smem_bytes_ont(P.wt, AMPO_WARPS, AMPO_GWARPS);
        if (!c->ont_attr) {
            CK(cudaFuncSetAttribute(amp_trim_pileup_ont_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(amp_trim_pileup_ont_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(amp_trim_pileup_ont_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            c->ont_attr = true;
        }
        P.gcap = P.tiles_per_cta;
        P.glist = glist;
        const bool tr = mode & AMP_MODE_TRIM, pl = mode & AMP_MODE_PILEUP;
        if (tr && pl) amp_trim_pileup_ont_kernel<true, true><<<grid, AMPO_WARPS * 32, smem, st>>>(P);
        else if (tr) amp_trim_pileup_ont_kernel<true, false><<<grid, AMPO_WARPS * 32, smem, st>>>(P);
        else amp_trim_pileup_ont_kernel<false, true><<<grid, AMPO_WARPS * 32, smem, st>>>(P);
        CK(cudaGetLastError());
        c->last_launches += 1;
        return AMP_OK;
    }
    P.wt = t.wt; P.maxseg = t.maxseg; P.qbytes = t.qbytes; P.sbytes = t.sbytes; P.reads_per_tile = t.reads_per_tile;
    P.ntiles = (int)((b.n + t.reads_per_tile - 1) / t.reads_per_tile);
    int grid = std::min(P.ntiles, c->sm_count * kCtasPerSm);
    P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
    grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
    const size_t smem = amp::smem_bytes(P.wt, P.maxseg, P.qbytes, P.sbytes);
    P.direct = t.direct;
    if (smem > c->max_dyn_smem) {
        CK(cudaFuncSetAttribute(amp_trim_pileup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaFuncSetAttribute(amp_trim_pileup_indel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        c->max_dyn_smem = smem;
    }
#ifdef AMP_PHASE_TIMING
    static long long* d_phase = nullptr;
    if (!d_phase) CK(cudaMalloc((void**)&d_phase, 4096 * 4 * 8));
    P.phase_cycles = d_phase;
#endif
    if (P.direct) amp_trim_pileup_indel_kernel<<<grid, kThreads, smem, st>>>(P);
    else amp_trim_pileup_kernel<<<grid, kThreads, smem, st>>>(P);
    CK(cudaGetLastError());
#ifdef AMP_PHASE_TIMING
    {
        CK(cudaStreamSynchronize(st));
        static long long h[4096 * 4];
        CK(cudaMemcpy(h, d_phase, sizeof(long long) * 4 * grid, cudaMemcpyDeviceToHost));
        double s4[4] = {0, 0, 0, 0};
        for (int b = 0; b < grid; ++b) for (int k = 0; k < 4; ++k) s4[k] += (double)h[b * 4 + k];
        fprintf(stderr, "[phase cycles per CTA, grid %d, tiles/CTA %d] S %.0f  T %.0f  W %.0f  C %.0f\n", grid, P.tiles_per_cta,
                s4[0] / grid, s4[1] / grid, s4[2] / grid, s4[3] / grid);
    }
#endif
    c->last_launches += 1;
    return AMP_OK;
}

// the fused kernel, then (AMP_MODE_QSTATS) the strand / quality pass over the same reads on the same stream
int launch_process(amp_ctx* c, const amp::BatchPtrs& b, long long sum_cig, long long max_cig, long long sum_qual, int mode,
                   int sample, const amp::TrimOut& o, uint32_t* scratch, uint32_t* glist, cudaStream_t st) {
    int rc = launch_fused(c, b, sum_cig, max_cig, sum_qual, mode, sample, o, scratch, glist, st);
    if (rc || !(mode & AMP_MODE_QSTATS) || b.n <= 0) return rc;
    amp::QStatsParams Q{};
    Q.b = b; Q.o = o; Q.trimmed = (mode & AMP_MODE_TRIM) ? 1 : 0;
    Q.L = c->cfg.ref_len;
    if ((size_t)sample < c->scheme.size() && c->scheme[sample].L > 0) Q.L = c->scheme[sample].L;   // as launch_fused
    Q.Lpad = c->Lpad; Q.minq = c->cfg.min_quality; Q.gpos_base = sample * c->Lpad;
    Q.rev = c->d_rev + (size_t)sample * AMP_NCH * c->Lpad; Q.qsum = c->d_qsum + (size_t)sample * AMP_NCH * c->Lpad;
    Q.tab = c->tab; Q.ins_rev = c->d_ins_rev; Q.ins_qsum = c->d_ins_qsum; Q.ins_head = c->d_ins_head; Q.err = c->d_err;
    const unsigned grid = (unsigned)((b.n + AMP_QS_READS - 1) / AMP_QS_READS);
    if (c->dels.slots) { Q.dels = c->dels; amp_qstats_dels_kernel<<<grid, AMP_QS_READS, 0, st>>>(Q); }
    else amp_qstats_kernel<<<grid, AMP_QS_READS, 0, st>>>(Q);
    CK(cudaGetLastError());
    c->last_launches += 1;
    return AMP_OK;
}

// AMP_MODE_QSTATS needs AMP_MODE_PILEUP and amp_qstats_enable
int check_qstats_mode(const amp_ctx* c, int mode, const char* who) {
    if (!(mode & AMP_MODE_QSTATS)) return AMP_OK;
    if (!(mode & AMP_MODE_PILEUP)) return fail(AMP_ERR_ARG, who, "AMP_MODE_QSTATS needs AMP_MODE_PILEUP");
    if (!c->d_rev) return fail(AMP_ERR_STATE, who, "AMP_MODE_QSTATS needs amp_qstats_enable first");
    return AMP_OK;
}

}  // namespace

extern "C" {

const char* amp_last_error(void) { return g_err.c_str(); }
int amp_abi_version(void) { return AMP_ABI_VERSION; }

int amp_create(const amp_config* cfg, const int32_t* min_primer_start, const int32_t* max_primer_end, int32_t max_primer_len,
               amp_ctx** out) {
    if (!cfg || !out || cfg->ref_len <= 0 || cfg->n_samples <= 0) return fail(AMP_ERR_ARG, "amp_create: bad config");
    if ((min_primer_start == nullptr) != (max_primer_end == nullptr)) return fail(AMP_ERR_ARG, "amp_create: need both primer tables or none");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(AMP_ERR_ARG, "amp_create: no such CUDA device");
    CK(cudaSetDevice(cfg->device));
    amp_ctx* c = new amp_ctx();
    c->cfg = *cfg;
    c->Lpad = (cfg->ref_len + 31) & ~31;
    c->max_primer_len = max_primer_len;
    CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, cfg->device));
    const size_t L = (size_t)cfg->ref_len;
    if (min_primer_start) {
        CK(cudaMalloc((void**)&c->d_min_start, L * 4));
        CK(cudaMalloc((void**)&c->d_max_end, L * 4));
        CK(cudaMemcpy(c->d_min_start, min_primer_start, L * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_max_end, max_primer_end, L * 4, cudaMemcpyHostToDevice));
    }
    CK(cudaMalloc((void**)&c->d_counts, (size_t)cfg->n_samples * AMP_NCH * c->Lpad * 4));
    unsigned long long nslots = cfg->ins_slots > 0 ? (unsigned long long)cfg->ins_slots : (1ULL << 21);
    while (nslots & (nslots - 1)) nslots += nslots & (~nslots + 1);   // round up to a power of two
    c->nslots = nslots;
    const unsigned long long arena_bytes = cfg->ins_arena_bytes > 0 ? (unsigned long long)cfg->ins_arena_bytes : (64ULL << 20);
    CK(cudaMalloc((void**)&c->tab.slots, nslots * sizeof(amp::InsSlot)));
    CK(cudaMalloc((void**)&c->tab.entries, nslots * 4));
    CK(cudaMalloc((void**)&c->tab.slot_entry, nslots * 4));
    CK(cudaMalloc((void**)&c->tab.arena, arena_bytes));
    CK(cudaMalloc((void**)&c->tab.cursor, 16));
    CK(cudaMalloc((void**)&c->d_err, 4));
    CK(cudaMalloc((void**)&c->tab.heads, (size_t)cfg->n_samples * c->Lpad * 4));
    CK(cudaMalloc((void**)&c->d_reset_done, 4));
    c->tab.mask = nslots - 1; c->tab.arena_words = arena_bytes / 8; c->tab.err = c->d_err;
    for (auto& ch : c->chunk) CK(cudaStreamCreateWithFlags(&ch.stream, cudaStreamNonBlocking));
    *out = c;
    int rc = amp_reset(c);
    if (rc) { amp_destroy(c); *out = nullptr; }
    return rc;
}

int amp_destroy(amp_ctx* c) {
    if (!c) return AMP_OK;
    cudaSetDevice(c->cfg.device);
    cudaDeviceSynchronize();
    cudaFree(c->d_min_start); cudaFree(c->d_max_end);
    for (auto& sc : c->scheme) { cudaFree(sc.d_min); cudaFree(sc.d_max); }
    if (c->counts_owned) cudaFree(c->d_counts);
    cudaFree(c->tab.slots); cudaFree(c->tab.entries); cudaFree(c->tab.slot_entry); cudaFree(c->tab.arena); cudaFree(c->tab.cursor); cudaFree(c->tab.heads);
    if (c->defl.stream) cudaStreamDestroy(c->defl.stream);
    cudaFree(c->defl.in); cudaFree(c->defl.slots); cudaFree(c->defl.out); cudaFree(c->defl.bstart); cudaFree(c->defl.off); cudaFree(c->defl.clen); cudaFree(c->defl.crc); cudaFree(c->defl.ctr); cudaFree(c->defl.toks);
    cudaFree(c->d_rev); cudaFree(c->d_qsum); cudaFree(c->d_ins_rev); cudaFree(c->d_ins_qsum); cudaFree(c->d_ins_head); cudaFree(c->d_ivar);
    cudaFree(c->dels.slots); cudaFree(c->dels.entries); cudaFree(c->dels.cursor); cudaFree(c->d_dels_out);
    cudaFree(c->d_err); cudaFree(c->d_reset_done); cudaFree(c->d_scratch); cudaFree(c->d_glist); cudaFree(c->d_ref); cudaFree(c->d_call); cudaFree(c->d_xbuf);
    {
        auto& d = c->dec;
        void* ps[] = {d.comp, d.raw, d.in_off, d.out_off, d.out_len, d.tot, d.prefix, d.ctr, d.pos, d.flag, d.tlen, d.cig_off, d.seq_off, d.qual_off,
                      d.rec_off, d.o_pos, d.o_ncig, d.o_flags, d.cigar, d.seq, d.qual, d.o_cigar, d.scratch, d.w_sizes, d.w_off, d.w_stream};
        for (void* q : ps) cudaFree(q);
        for (auto& e : d.ev) if (e) cudaEventDestroy(e);
        for (auto& z : d.zs) if (z) cudaStreamDestroy(z);
    }
    {
        auto& t = c->ct;
        void* ps[] = {t.sid, t.hist, t.hist_off, t.table, t.perm, t.tsum, t.tbase, t.pos, t.flag, t.tlen, t.cig_off, t.seq_off, t.qual_off, t.cigar,
                      t.seq, t.qual, t.o_pos, t.o_ncig, t.o_flags, t.o_cigar, t.scratch};
        for (void* q : ps) cudaFree(q);
    }
    cudaFree(c->an.tables); cudaFree(c->an.off); cudaFree(c->an.tsum); cudaFree(c->an.tbase); cudaFree(c->an.e_int); cudaFree(c->an.e_chr);
    for (auto& ch : c->chunk) {
        cudaFree(ch.pos); cudaFree(ch.flag); cudaFree(ch.tlen); cudaFree(ch.cig_off); cudaFree(ch.seq_off); cudaFree(ch.qual_off);
        cudaFree(ch.cigar); cudaFree(ch.seq); cudaFree(ch.qual); cudaFree(ch.o_pos); cudaFree(ch.o_ncig); cudaFree(ch.o_flags);
        cudaFree(ch.o_cigar); cudaFree(ch.scratch); cudaFree(ch.glist);
        if (ch.stream) cudaStreamDestroy(ch.stream);
    }
    delete c;
    return AMP_OK;
}

int amp_reset(amp_ctx* c) {
    if (!c) return fail(AMP_ERR_ARG, "amp_reset: null context");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaMemsetAsync(c->d_counts, 0, (size_t)c->cfg.n_samples * AMP_NCH * c->Lpad * 4, 0));
    CK(cudaMemsetAsync(c->tab.slots, 0, c->nslots * sizeof(amp::InsSlot), 0));
    CK(cudaMemsetAsync(c->tab.heads, 0xFF, (size_t)c->cfg.n_samples * c->Lpad * 4, 0));
    CK(cudaMemsetAsync(c->tab.cursor, 0, 16, 0));
    CK(cudaMemsetAsync(c->d_err, 0, 4, 0));
    CK(cudaMemsetAsync(c->d_reset_done, 0, 4, 0));
    if (c->d_rev) {
        const size_t n = (size_t)c->cfg.n_samples * AMP_NCH * c->Lpad;
        CK(cudaMemsetAsync(c->d_rev, 0, n * 4, 0)); CK(cudaMemsetAsync(c->d_qsum, 0, n * 8, 0));
        CK(cudaMemsetAsync(c->d_ins_rev, 0, c->nslots * 4, 0)); CK(cudaMemsetAsync(c->d_ins_qsum, 0, c->nslots * 8, 0));
        CK(cudaMemsetAsync(c->d_ins_head, 0, c->nslots, 0));
    }
    if (c->dels.slots) {
        CK(cudaMemsetAsync(c->dels.slots, 0, c->dels_nslots * sizeof(amp::DelSlot), 0));
        CK(cudaMemsetAsync(c->dels.cursor, 0, 8, 0));
    }
    CK(cudaStreamSynchronize(0));
    return AMP_OK;
}

int amp_reset_async(amp_ctx* c, void* stream) {
    if (!c) return fail(AMP_ERR_ARG, "amp_reset_async: null context");
    CK(cudaSetDevice(c->cfg.device));
    // counts: n_samples * 6 * Lpad ints and heads: n_samples * Lpad ints, Lpad a multiple of 32 -- whole 16-byte words
    const unsigned long long counts16 = (unsigned long long)c->cfg.n_samples * AMP_NCH * c->Lpad / 4;
    const unsigned long long heads16 = (unsigned long long)c->cfg.n_samples * c->Lpad / 4;
    const unsigned long long grid = std::min<unsigned long long>((counts16 + 255) / 256, (unsigned long long)c->sm_count * 8);
    auto* k = c->d_rev ? amp_reset_kernel<true> : amp_reset_kernel<false>;
    k<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((uint4*)c->d_counts, counts16, (uint4*)c->tab.heads, heads16, c->tab.slots, c->tab.entries,
                                                        c->tab.cursor, c->d_err, c->d_reset_done, (uint4*)c->d_rev, (uint4*)c->d_qsum, counts16,
                                                        c->d_ins_rev, c->d_ins_qsum, c->d_ins_head);
    CK(cudaGetLastError());
    if (c->dels.slots) {
        amp_dels_reset_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(c->dels);
        CK(cudaGetLastError());
    }
    return AMP_OK;
}

int amp_error_flags(amp_ctx* c, uint32_t* flags) {
    if (!c || !flags) return fail(AMP_ERR_ARG, "amp_error_flags: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(flags, c->d_err, 4, cudaMemcpyDeviceToHost));
    return AMP_OK;
}

int amp_lpad(amp_ctx* c) { return c ? c->Lpad : AMP_ERR_ARG; }
int amp_sm_count(amp_ctx* c) { return c ? c->sm_count : AMP_ERR_ARG; }
int amp_last_launches(amp_ctx* c) { return c ? c->last_launches : AMP_ERR_ARG; }

int amp_process_device(amp_ctx* c, const amp_batch* b, int64_t sum_cigar_ops, int64_t sum_qual_bytes, int mode, int sample,
                       const amp_trim_out* o, void* stream) {
    if (!c || !b) return fail(AMP_ERR_ARG, "amp_process_device: null argument");
    if (sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_process_device: sample out of range");
    if ((mode & AMP_MODE_TRIM) && (!o || !has_scheme(c, sample))) return fail(AMP_ERR_ARG, "amp_process_device: trimming needs primer tables and an output block");
    if (!(mode & (AMP_MODE_TRIM | AMP_MODE_PILEUP))) return fail(AMP_ERR_ARG, "amp_process_device: empty mode");
    if (int rc = check_qstats_mode(c, mode, "amp_process_device")) return rc;
    CK(cudaSetDevice(c->cfg.device));
    c->last_launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (mode & AMP_MODE_TRIM) {
        // long-CIGAR scratch (2 rows per read); allocated once per high-water mark
        const size_t need = 2 * ((size_t)sum_cigar_ops + 3 * (size_t)b->n_reads);
        if (need > c->scratch_words) {
            CK(cudaStreamSynchronize(st));
            if (c->d_scratch) CK(cudaFree(c->d_scratch));
            c->d_scratch = nullptr; c->scratch_words = 0;
            CK(cudaMalloc((void**)&c->d_scratch, need * 4));
            c->scratch_words = need;
        }
    }
    {
        const size_t need = glist_words_for(c, b->n_reads);
        if (need > c->glist_words) {
            CK(cudaStreamSynchronize(st));
            if (c->d_glist) CK(cudaFree(c->d_glist));
            c->d_glist = nullptr; c->glist_words = 0;
            CK(cudaMalloc((void**)&c->d_glist, need * 4));
            c->glist_words = need;
        }
    }
    amp::BatchPtrs bp{b->first, b->n_reads, b->pos, b->flag, b->tlen, b->cig_off, b->cigar, b->seq_off, b->seq, b->qual_off, b->qual};
    amp::TrimOut to{};
    if (o) { to.pos = o->pos; to.ncig = o->ncig; to.flags = o->flags; to.cigar = o->cigar; }
    uint32_t* scratch = c->d_scratch;
    if ((mode & AMP_MODE_TRIM) && b->first != 0) {   // scratch rows are addressed like the output rows: shift to the range start
        uint32_t c_first = 0;
        CK(cudaMemcpyAsync(&c_first, b->cig_off + b->first, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        scratch -= (size_t)c_first + 3 * (size_t)b->first;
    }
    if (sum_qual_bytes <= 0) sum_qual_bytes = (long long)b->n_reads * 150;
    return launch_process(c, bp, sum_cigar_ops, 0, sum_qual_bytes, mode, sample, to, scratch, c->d_glist, st);
}

int amp_process_host(amp_ctx* c, const amp_batch* b, int mode, int sample, const amp_trim_out* o) {
    if (!c || !b) return fail(AMP_ERR_ARG, "amp_process_host: null argument");
    if (sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_process_host: sample out of range");
    if ((mode & AMP_MODE_TRIM) && (!o || !has_scheme(c, sample))) return fail(AMP_ERR_ARG, "amp_process_host: trimming needs primer tables and an output block");
    if (!(mode & (AMP_MODE_TRIM | AMP_MODE_PILEUP))) return fail(AMP_ERR_ARG, "amp_process_host: empty mode");
    if (int rc = check_qstats_mode(c, mode, "amp_process_host")) return rc;
    CK(cudaSetDevice(c->cfg.device));
    c->last_launches = 0;
    const bool trim = mode & AMP_MODE_TRIM, pile = mode & AMP_MODE_PILEUP;
    const long long first = b->first, last = b->first + b->n_reads;
    const long long kChunk = 1 << 18;   // reads per in-flight chunk: three of them keep both copy engines and the SMs busy
    int slot = 0;
    for (long long a = first; a < last; a += kChunk, slot = (slot + 1) % 3) {
        const long long e = std::min(last, a + kChunk), n = e - a;
        DevChunk& d = c->chunk[slot];
        CK(cudaStreamSynchronize(d.stream));   // previous use of this slot has drained
        const size_t c0 = b->cig_off[a], c1 = b->cig_off[e];
        const size_t q0 = b->qual_off[a] & ~(size_t)15, q1 = b->qual_off[e];
        const size_t s0 = b->seq_off[a] & ~(size_t)15, s1 = b->seq_off[e];
        if ((size_t)n + 1 > d.cap_reads) {
            const size_t want = (size_t)n + 1 + 64;
            void** arrs[9] = {(void**)&d.pos, (void**)&d.flag, (void**)&d.tlen, (void**)&d.cig_off, (void**)&d.seq_off,
                              (void**)&d.qual_off, (void**)&d.o_pos, (void**)&d.o_ncig, (void**)&d.o_flags};
            for (void** ap : arrs) {
                if (*ap) CK(cudaFree(*ap));
                *ap = nullptr;
                CK(cudaMalloc(ap, want * 4));
            }
            d.cap_reads = want;
        }
        {
            int rc;
            if ((rc = dev_grow(&d.cigar, &d.cap_cig, (c1 - c0) + 4))) return rc;
            if ((rc = dev_grow(&d.qual, &d.cap_qual, (q1 - q0) + 32))) return rc;
            if ((rc = dev_grow(&d.glist, &d.cap_glist, glist_words_for(c, n)))) return rc;
            if (pile && (rc = dev_grow(&d.seq, &d.cap_seq, (s1 - s0) + 32))) return rc;
            if (trim) {
                const size_t orows = (c1 - c0) + 3 * (size_t)n;
                if ((rc = dev_grow(&d.o_cigar, &d.cap_ocigar, orows + 4))) return rc;
                // the two global scratch rows per read are only touched by CIGARs too long for the kernels' on-chip rows;
                // they are allocated regardless (a scan of the chunk for its longest CIGAR would sit in front of the copies)
                if ((rc = dev_grow(&d.scratch, &d.cap_scratch, 2 * (orows + 4)))) return rc;
            }
        }
        cudaStream_t st = d.stream;
        CK(cudaMemcpyAsync(d.pos, b->pos + a, n * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d.flag, b->flag + a, n * 2, cudaMemcpyHostToDevice, st));
        if (trim) CK(cudaMemcpyAsync(d.tlen, b->tlen + a, n * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d.cig_off, b->cig_off + a, (n + 1) * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d.qual_off, b->qual_off + a, (n + 1) * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d.seq_off, b->seq_off + a, (n + 1) * 4, cudaMemcpyHostToDevice, st));
        if (c1 > c0) CK(cudaMemcpyAsync(d.cigar, b->cigar + c0, (c1 - c0) * 4, cudaMemcpyHostToDevice, st));
        if (q1 > q0) CK(cudaMemcpyAsync(d.qual, b->qual + q0, q1 - q0, cudaMemcpyHostToDevice, st));
        if (pile && s1 > s0) CK(cudaMemcpyAsync(d.seq, b->seq + s0, s1 - s0, cudaMemcpyHostToDevice, st));
        // pointers are indexed with global read indices / absolute offsets: shift the chunk buffers back
        amp::BatchPtrs bp{a, n, d.pos - a, d.flag - a, d.tlen - a, d.cig_off - a, d.cigar - c0, d.seq_off - a,
                          pile ? d.seq - s0 : nullptr, d.qual_off - a, d.qual - q0};
        amp::TrimOut to{};
        const size_t orow0 = c0 + 3 * (size_t)a;
        if (trim) { to.pos = d.o_pos - a; to.ncig = d.o_ncig - a; to.flags = d.o_flags - a; to.cigar = d.o_cigar - orow0; }
        int rc = launch_process(c, bp, (long long)(c1 - c0), 0, (long long)(b->qual_off[e] - b->qual_off[a]), mode, sample, to,
                                (trim && d.scratch) ? d.scratch - orow0 : nullptr, d.glist, st);
        if (rc) return rc;
        if (trim) {
            CK(cudaMemcpyAsync(o->pos + a, d.o_pos, n * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(o->ncig + a, d.o_ncig, n * 2, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(o->flags + a, d.o_flags, n, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(o->cigar + orow0, d.o_cigar, ((c1 - c0) + 3 * (size_t)n) * 4, cudaMemcpyDeviceToHost, st));
        }
    }
    for (auto& ch : c->chunk) CK(cudaStreamSynchronize(ch.stream));
    return AMP_OK;
}

int amp_counts_device(amp_ctx* c, int32_t** dev_counts) {
    if (!c || !dev_counts) return fail(AMP_ERR_ARG, "amp_counts_device: null argument");
    *dev_counts = c->d_counts;
    return AMP_OK;
}

int amp_bind_counts(amp_ctx* c, int32_t* dev_counts) {
    if (!c || !dev_counts) return fail(AMP_ERR_ARG, "amp_bind_counts: null argument");
    if ((uintptr_t)dev_counts & 15) return fail(AMP_ERR_ARG, "amp_bind_counts: the buffer must be 16-byte aligned");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    if (c->counts_owned) CK(cudaFree(c->d_counts));
    c->d_counts = dev_counts; c->counts_owned = false;
    return AMP_OK;
}

int amp_counts_host(amp_ctx* c, int sample, int32_t* host) {
    if (!c || !host || sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_counts_host: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t L = (size_t)c->cfg.ref_len;
    CK(cudaMemcpy2D(host, L * 4, c->d_counts + (size_t)sample * AMP_NCH * c->Lpad, (size_t)c->Lpad * 4, L * 4, AMP_NCH,
                    cudaMemcpyDeviceToHost));
    return AMP_OK;
}

// the inverse of amp_counts_host: replace count matrix `sample` by host values (function-level drop-ins, tests)
int amp_counts_upload(amp_ctx* c, int sample, const int32_t* host) {
    if (!c || !host || sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_counts_upload: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t L = (size_t)c->cfg.ref_len;
    CK(cudaMemset(c->d_counts + (size_t)sample * AMP_NCH * c->Lpad, 0, (size_t)AMP_NCH * c->Lpad * 4));
    CK(cudaMemcpy2D(c->d_counts + (size_t)sample * AMP_NCH * c->Lpad, (size_t)c->Lpad * 4, host, L * 4, L * 4, AMP_NCH, cudaMemcpyHostToDevice));
    return AMP_OK;
}

int amp_ins_count(amp_ctx* c, int64_t* n_alleles, int64_t* n_chars) {
    if (!c || !n_alleles || !n_chars) return fail(AMP_ERR_ARG, "amp_ins_count: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    unsigned long long cur[2];
    CK(cudaMemcpy(cur, c->tab.cursor, 16, cudaMemcpyDeviceToHost));
    *n_alleles = (int64_t)cur[1];
    *n_chars = (int64_t)(std::min(cur[0], c->tab.arena_words) * 8);   // upper bound (records incl. headers and padding)
    return AMP_OK;
}

int amp_ins_export(amp_ctx* c, int32_t* sample, int32_t* pos, int32_t* count, int64_t* str_off, char* chars) {
    if (!c || !str_off) return fail(AMP_ERR_ARG, "amp_ins_export: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    unsigned long long cur[2];
    CK(cudaMemcpy(cur, c->tab.cursor, 16, cudaMemcpyDeviceToHost));
    const unsigned long long n = cur[1];
    // a failed reservation leaves cursor[0] past the arena (AMP_E_ARENA_FULL); the stored records all lie below arena_words
    const unsigned long long words = std::min(cur[0], c->tab.arena_words);
    str_off[0] = 0;
    if (n == 0) return AMP_OK;
    {
        int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n * 16 + 64);
        if (rc) return rc;
    }
    unsigned long long* d_off = (unsigned long long*)c->d_xbuf;
    int* d_count = (int*)(c->d_xbuf + (size_t)n * 8);
    amp_gather_entries_kernel<<<(unsigned)std::min<unsigned long long>((n + 255) / 256, 1184), 256>>>(c->tab.slots, c->tab.entries, n, d_count, d_off);
    CK(cudaGetLastError());
    std::vector<unsigned long long> off(n);
    std::vector<unsigned char> arena(words * 8);
    CK(cudaMemcpy(count, d_count, n * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(off.data(), d_off, n * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(arena.data(), c->tab.arena, words * 8, cudaMemcpyDeviceToHost));
    int64_t o = 0;
    for (unsigned long long k = 0; k < n; ++k) {
        const unsigned char* rec = arena.data() + off[k] * 8;
        int gpos; unsigned int len;
        memcpy(&gpos, rec, 4); memcpy(&len, rec + 4, 4);
        sample[k] = gpos / c->Lpad; pos[k] = gpos % c->Lpad;
        memcpy(chars + o, rec + 8, len);
        o += len; str_off[k + 1] = o;
    }
    return AMP_OK;
}

int amp_ins_merge(amp_ctx* c, int64_t n, const int32_t* sample, const int32_t* pos, const int32_t* count, const int64_t* str_off,
                  const char* chars) {
    if (!c || n < 0) return fail(AMP_ERR_ARG, "amp_ins_merge: bad argument");
    if (n == 0) return AMP_OK;
    CK(cudaSetDevice(c->cfg.device));
    std::vector<int> gpos(n);
    for (int64_t k = 0; k < n; ++k) gpos[k] = sample[k] * c->Lpad + pos[k];
    const size_t nch = (size_t)str_off[n];
    const size_t o_count = (size_t)n * 4, o_off = ((size_t)n * 8 + 7) & ~(size_t)7, o_chars = o_off + ((size_t)n + 1) * 8;
    {
        int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, o_chars + nch + 64);
        if (rc) return rc;
    }
    int* d_gpos = (int*)c->d_xbuf; int* d_count = (int*)(c->d_xbuf + o_count);
    long long* d_off = (long long*)(c->d_xbuf + o_off); char* d_chars = (char*)(c->d_xbuf + o_chars);
    CK(cudaMemcpy(d_gpos, gpos.data(), n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_count, count, n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_off, str_off, (n + 1) * 8, cudaMemcpyHostToDevice));
    if (nch) CK(cudaMemcpy(d_chars, chars, nch, cudaMemcpyHostToDevice));
    amp_merge_kernel<<<(unsigned)std::min<int64_t>((n + 127) / 128, 1184), 128>>>(c->tab, n, d_gpos, d_count, d_off, d_chars);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return AMP_OK;
}

int amp_set_reference(amp_ctx* c, const char* ref_seq) {
    if (!c || !ref_seq) return fail(AMP_ERR_ARG, "amp_set_reference: null argument");
    CK(cudaSetDevice(c->cfg.device));
    if (c->ref_per_sample) { CK(cudaFree(c->d_ref)); c->d_ref = nullptr; c->ref_per_sample = false; c->ref_len_s.clear(); }
    c->an.built = false;
    if (!c->d_ref) CK(cudaMalloc((void**)&c->d_ref, (size_t)c->cfg.ref_len + 16));
    CK(cudaMemcpy(c->d_ref, ref_seq, (size_t)c->cfg.ref_len, cudaMemcpyHostToDevice));
    return AMP_OK;
}

// device-side calling: outputs stay in context-owned HBM buffers; asynchronous on `stream`
int amp_call_device(amp_ctx* c, const amp_call_params* p, void* stream) {
    if (!c || !p) return fail(AMP_ERR_ARG, "amp_call_device: null argument");
    if (!c->d_ref) return fail(AMP_ERR_STATE, "amp_call_device: amp_set_reference has not been called");
    CK(cudaSetDevice(c->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t L = (size_t)c->cfg.ref_len, S = (size_t)c->cfg.n_samples, SL = S * L;
    if (!c->d_call) {
        size_t bytes = 0;
        auto take = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
        c->o_depth = take(SL * 4); c->o_top = take(SL * 4); c->o_topc = take(SL * 4); c->o_fl = take(SL); c->o_refc = take(SL * 4);
        c->o_ff = take(SL * 6 * 8); c->o_fr = take(SL * 6 * 4); c->o_alt = take(SL);
        c->o_if = take(c->nslots * 8); c->o_ir = take(c->nslots * 4); c->o_ia = take(c->nslots);
        CK(cudaMalloc((void**)&c->d_call, bytes + 256));
    }
    c->last_launches = 0;
    unsigned char* blk = c->d_call;
    amp::CallParams P{};
    P.L = (int)L; P.Lpad = c->Lpad; P.n_samples = (int)S; P.counts = c->d_counts; P.slots = c->tab.slots;
    P.slot_entry = c->tab.slot_entry; P.arena = c->tab.arena; P.heads = c->tab.heads; P.ref_seq = c->d_ref;
    P.ref_stride = c->ref_per_sample ? (long long)c->cfg.ref_len : 0;
    P.min_depth_consensus = p->min_depth_consensus; P.min_freq_consensus = p->min_freq_consensus;
    P.min_depth_variants = p->min_depth_variants; P.min_freq_variants = p->min_freq_variants;
    P.depth = (int*)(blk + c->o_depth); P.top_id = (int*)(blk + c->o_top); P.top_count = (int*)(blk + c->o_topc);
    P.pos_flags = blk + c->o_fl; P.ref_count = (int*)(blk + c->o_refc); P.fixed_freq = (double*)(blk + c->o_ff);
    P.fixed_rank = (int*)(blk + c->o_fr); P.alt_mask = blk + c->o_alt; P.ins_freq = (double*)(blk + c->o_if);
    P.ins_rank = (int*)(blk + c->o_ir); P.ins_alt = blk + c->o_ia;
    // the insertion lists are current: ins_table_add links every allele it creates
    amp_call_kernel<<<(unsigned)((SL * AMP_CALL_LANES + 255) / 256), 256, 0, st>>>(P);
    CK(cudaGetLastError());
    c->last_launches = 1;
    return AMP_OK;
}

int amp_call(amp_ctx* c, const char* ref_seq, const amp_call_params* p, const amp_call_out* ho, double* ins_freq,
             int32_t* ins_rank, uint8_t* ins_alt) {
    if (!c || !p || !ho) return fail(AMP_ERR_ARG, "amp_call: null argument");
    int rc;
    if (ref_seq && (rc = amp_set_reference(c, ref_seq))) return rc;
    CK(cudaDeviceSynchronize());
    cudaStream_t st = c->chunk[0].stream;   // idle after the synchronize; copies queue behind the kernels on it
    if ((rc = amp_call_device(c, p, st))) return rc;
    const size_t L = (size_t)c->cfg.ref_len, S = (size_t)c->cfg.n_samples, SL = S * L;
    unsigned long long cur[2];
    CK(cudaMemcpyAsync(cur, c->tab.cursor, 16, cudaMemcpyDeviceToHost, st));
    unsigned char* blk = c->d_call;
    // one queue of asynchronous copies and one wait: with page-locked destinations (amp_host_alloc) they run back to back
    if (ho->depth) CK(cudaMemcpyAsync(ho->depth, blk + c->o_depth, SL * 4, cudaMemcpyDeviceToHost, st));
    if (ho->top_id) CK(cudaMemcpyAsync(ho->top_id, blk + c->o_top, SL * 4, cudaMemcpyDeviceToHost, st));
    if (ho->top_count) CK(cudaMemcpyAsync(ho->top_count, blk + c->o_topc, SL * 4, cudaMemcpyDeviceToHost, st));
    if (ho->pos_flags) CK(cudaMemcpyAsync(ho->pos_flags, blk + c->o_fl, SL, cudaMemcpyDeviceToHost, st));
    if (ho->ref_count) CK(cudaMemcpyAsync(ho->ref_count, blk + c->o_refc, SL * 4, cudaMemcpyDeviceToHost, st));
    if (ho->fixed_freq) CK(cudaMemcpyAsync(ho->fixed_freq, blk + c->o_ff, SL * 6 * 8, cudaMemcpyDeviceToHost, st));
    if (ho->fixed_rank) CK(cudaMemcpyAsync(ho->fixed_rank, blk + c->o_fr, SL * 6 * 4, cudaMemcpyDeviceToHost, st));
    if (ho->alt_mask) CK(cudaMemcpyAsync(ho->alt_mask, blk + c->o_alt, SL, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const size_t K = (size_t)cur[1];
    if (K && ins_freq) CK(cudaMemcpyAsync(ins_freq, blk + c->o_if, K * 8, cudaMemcpyDeviceToHost, st));
    if (K && ins_rank) CK(cudaMemcpyAsync(ins_rank, blk + c->o_ir, K * 4, cudaMemcpyDeviceToHost, st));
    if (K && ins_alt) CK(cudaMemcpyAsync(ins_alt, blk + c->o_ia, K, cudaMemcpyDeviceToHost, st));
    if (K) CK(cudaStreamSynchronize(st));
    return AMP_OK;
}

int amp_qstats_enable(amp_ctx* c) {
    if (!c) return fail(AMP_ERR_ARG, "amp_qstats_enable: null context");
    if (c->d_rev) return AMP_OK;
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t n = (size_t)c->cfg.n_samples * AMP_NCH * c->Lpad;
    CK(cudaMalloc((void**)&c->d_rev, n * 4)); CK(cudaMalloc((void**)&c->d_qsum, n * 8));
    CK(cudaMalloc((void**)&c->d_ins_rev, c->nslots * 4)); CK(cudaMalloc((void**)&c->d_ins_qsum, c->nslots * 8));
    CK(cudaMalloc((void**)&c->d_ins_head, c->nslots));
    CK(cudaMemset(c->d_rev, 0, n * 4)); CK(cudaMemset(c->d_qsum, 0, n * 8));
    CK(cudaMemset(c->d_ins_rev, 0, c->nslots * 4)); CK(cudaMemset(c->d_ins_qsum, 0, c->nslots * 8)); CK(cudaMemset(c->d_ins_head, 0, c->nslots));
    return AMP_OK;
}

int amp_qstats_host(amp_ctx* c, int sample, int32_t* rev, int64_t* qsum, int32_t* ins_rev, int64_t* ins_qsum, uint8_t* ins_head) {
    if (!c || sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_qstats_host: bad argument");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_qstats_host: amp_qstats_enable has not been called");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t L = (size_t)c->cfg.ref_len, base = (size_t)sample * AMP_NCH * c->Lpad;
    if (rev) CK(cudaMemcpy2D(rev, L * 4, c->d_rev + base, (size_t)c->Lpad * 4, L * 4, AMP_NCH, cudaMemcpyDeviceToHost));
    if (qsum) CK(cudaMemcpy2D(qsum, L * 8, c->d_qsum + base, (size_t)c->Lpad * 8, L * 8, AMP_NCH, cudaMemcpyDeviceToHost));
    unsigned long long cur[2];
    CK(cudaMemcpy(cur, c->tab.cursor, 16, cudaMemcpyDeviceToHost));
    const unsigned long long n = cur[1];
    if (n == 0 || !(ins_rev || ins_qsum || ins_head)) return AMP_OK;
    {
        int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n * 13 + 64);
        if (rc) return rc;
    }
    unsigned long long* d_q = (unsigned long long*)c->d_xbuf;
    int* d_r = (int*)(c->d_xbuf + (size_t)n * 8);
    unsigned char* d_h = c->d_xbuf + (size_t)n * 12;
    amp_qstats_gather_kernel<<<(unsigned)std::min<unsigned long long>((n + 255) / 256, 1184), 256>>>(c->tab.entries, n, c->d_ins_rev, c->d_ins_qsum,
                                                                                                    c->d_ins_head, d_r, d_q, d_h);
    CK(cudaGetLastError());
    if (ins_rev) CK(cudaMemcpy(ins_rev, d_r, n * 4, cudaMemcpyDeviceToHost));
    if (ins_qsum) CK(cudaMemcpy(ins_qsum, d_q, n * 8, cudaMemcpyDeviceToHost));
    if (ins_head) CK(cudaMemcpy(ins_head, d_h, n, cudaMemcpyDeviceToHost));
    return AMP_OK;
}

// device-side iVar calling on the outputs amp_call_device left in the context; asynchronous on `stream`
int amp_call_ivar_device(amp_ctx* c, const amp_ivar_params* p, void* stream) {
    if (!c || !p) return fail(AMP_ERR_ARG, "amp_call_ivar_device: null argument");
    if (!(p->iupac_threshold >= 0.0 && p->iupac_threshold <= 1.0)) return fail(AMP_ERR_ARG, "amp_call_ivar_device: iupac_threshold must be in [0, 1]");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_call_ivar_device: amp_qstats_enable has not been called");
    if (!c->d_call) return fail(AMP_ERR_STATE, "amp_call_ivar_device: amp_call / amp_call_device has not been called");
    CK(cudaSetDevice(c->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t L = (size_t)c->cfg.ref_len, S = (size_t)c->cfg.n_samples, SL = S * L;
    if (!c->d_ivar) {
        size_t bytes = 0;
        auto take = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
        c->o_iu = take(SL); c->o_fmq = take(SL * 6 * 4); c->o_fpv = take(SL * 6 * 8); c->o_imq = take(c->nslots * 4); c->o_ipv = take(c->nslots * 8);
        CK(cudaMalloc((void**)&c->d_ivar, bytes + 256));
    }
    unsigned char* blk = c->d_call;
    unsigned char* out = c->d_ivar;
    amp::IvarParams P{};
    P.L = (int)L; P.Lpad = c->Lpad; P.n_samples = (int)S; P.counts = c->d_counts; P.qsum = c->d_qsum;
    P.slots = c->tab.slots; P.slot_entry = c->tab.slot_entry; P.arena = c->tab.arena; P.heads = c->tab.heads; P.ins_qsum = c->d_ins_qsum;
    P.ref_seq = c->d_ref; P.ref_stride = c->ref_per_sample ? (long long)c->cfg.ref_len : 0;
    P.depth = (const int*)(blk + c->o_depth); P.top_id = (const int*)(blk + c->o_top); P.top_count = (const int*)(blk + c->o_topc);
    P.fixed_freq = (const double*)(blk + c->o_ff); P.fixed_rank = (const int*)(blk + c->o_fr);
    P.ins_freq = (const double*)(blk + c->o_if); P.ins_rank = (const int*)(blk + c->o_ir);
    P.min_depth = p->min_depth; P.min_freq = p->min_freq; P.iupac_threshold = p->iupac_threshold;
    P.iupac = out + c->o_iu; P.fixed_mq = (int*)(out + c->o_fmq); P.fixed_pval = (double*)(out + c->o_fpv);
    P.ins_mq = (int*)(out + c->o_imq); P.ins_pval = (double*)(out + c->o_ipv);
    amp_ivar_kernel<<<(unsigned)((SL + 255) / 256), 256, 0, st>>>(P);
    CK(cudaGetLastError());
    c->last_launches = 1;
    return AMP_OK;
}

int amp_call_ivar(amp_ctx* c, const amp_ivar_params* p, uint8_t* iupac, int32_t* fixed_mq, double* fixed_pval, int32_t* ins_mq,
                  double* ins_pval) {
    if (!c || !p) return fail(AMP_ERR_ARG, "amp_call_ivar: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    cudaStream_t st = c->chunk[0].stream;
    int rc;
    if ((rc = amp_call_ivar_device(c, p, st))) return rc;
    const size_t SL = (size_t)c->cfg.n_samples * c->cfg.ref_len;
    unsigned long long cur[2];
    CK(cudaMemcpyAsync(cur, c->tab.cursor, 16, cudaMemcpyDeviceToHost, st));
    unsigned char* out = c->d_ivar;
    if (iupac) CK(cudaMemcpyAsync(iupac, out + c->o_iu, SL, cudaMemcpyDeviceToHost, st));
    if (fixed_mq) CK(cudaMemcpyAsync(fixed_mq, out + c->o_fmq, SL * 6 * 4, cudaMemcpyDeviceToHost, st));
    if (fixed_pval) CK(cudaMemcpyAsync(fixed_pval, out + c->o_fpv, SL * 6 * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const size_t K = (size_t)cur[1];
    if (K && ins_mq) CK(cudaMemcpyAsync(ins_mq, out + c->o_imq, K * 4, cudaMemcpyDeviceToHost, st));
    if (K && ins_pval) CK(cudaMemcpyAsync(ins_pval, out + c->o_ipv, K * 8, cudaMemcpyDeviceToHost, st));
    if (K) CK(cudaStreamSynchronize(st));
    return AMP_OK;
}

// ---- anchored deletion alleles (amp_dels.cuh) ------------------------------------------------------------------------------------
int amp_dels_enable(amp_ctx* c, int64_t slots) {
    if (!c || slots < 0 || slots > (1LL << 40)) return fail(AMP_ERR_ARG, "amp_dels_enable: bad argument");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_dels_enable: amp_qstats_enable has not been called (the strand / quality pass fills the table)");
    if (c->dels.slots) return AMP_OK;
    unsigned long long n = slots > 0 ? (unsigned long long)slots : (1ULL << 20);
    while (n & (n - 1)) n += n & (~n + 1);   // round up to a power of two
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    CK(cudaMalloc((void**)&c->dels.slots, n * sizeof(amp::DelSlot)));
    CK(cudaMalloc((void**)&c->dels.entries, n * 4));
    CK(cudaMalloc((void**)&c->dels.cursor, 8));
    CK(cudaMemset(c->dels.slots, 0, n * sizeof(amp::DelSlot)));
    CK(cudaMemset(c->dels.cursor, 0, 8));
    c->dels.mask = n - 1; c->dels.err = c->d_err; c->dels_nslots = n;
    return AMP_OK;
}

static int dels_check(amp_ctx* c, const char* who) {
    if (!c) return fail(AMP_ERR_ARG, who, "null context");
    if (!c->dels.slots) return fail(AMP_ERR_STATE, who, "amp_dels_enable has not been called");
    return AMP_OK;
}
// the listed alleles on the host: {key, count | rev << 32, qsum} per allele, and the list order sorted by key
static int dels_download(amp_ctx* c, std::vector<unsigned long long>& rec, std::vector<unsigned long long>& order) {
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    unsigned long long n = 0;
    CK(cudaMemcpy(&n, c->dels.cursor, 8, cudaMemcpyDeviceToHost));
    rec.assign(3 * n, 0); order.resize(n);
    for (unsigned long long k = 0; k < n; ++k) order[k] = k;
    if (n == 0) return AMP_OK;
    if (int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n * 24 + 64)) return rc;
    amp_dels_gather_kernel<<<(unsigned)std::min<unsigned long long>((n + 255) / 256, 1184), 256>>>(c->dels, n, (unsigned long long*)c->d_xbuf);
    CK(cudaGetLastError());
    CK(cudaMemcpy(rec.data(), c->d_xbuf, n * 24, cudaMemcpyDeviceToHost));
    // LSD radix sort by key, 16 bits a pass; a pass whose digit is the same for every key is skipped (the high bits of a length)
    std::vector<unsigned long long> tmp(n);
    std::vector<size_t> hist(1 << 16);
    for (int shift = 0; shift < 64; shift += 16) {
        std::fill(hist.begin(), hist.end(), 0);
        for (unsigned long long k = 0; k < n; ++k) ++hist[(rec[3 * order[k]] >> shift) & 0xFFFF];
        if (hist[(rec[0] >> shift) & 0xFFFF] == n) continue;
        size_t sum = 0;
        for (auto& h : hist) { const size_t t = h; h = sum; sum += t; }
        for (unsigned long long k = 0; k < n; ++k) tmp[hist[(rec[3 * order[k]] >> shift) & 0xFFFF]++] = order[k];
        order.swap(tmp);
    }
    return AMP_OK;
}

int amp_dels_count(amp_ctx* c, int64_t* n) {
    if (int rc = dels_check(c, "amp_dels_count")) return rc;
    if (!n) return fail(AMP_ERR_ARG, "amp_dels_count: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    unsigned long long v = 0;
    CK(cudaMemcpy(&v, c->dels.cursor, 8, cudaMemcpyDeviceToHost));
    *n = (int64_t)v;
    return AMP_OK;
}

int amp_dels_export(amp_ctx* c, int32_t* sample, int32_t* anchor, int32_t* len, int32_t* count, int32_t* rev, int64_t* qsum) {
    if (int rc = dels_check(c, "amp_dels_export")) return rc;
    std::vector<unsigned long long> rec, order;
    if (int rc = dels_download(c, rec, order)) return rc;
    for (size_t j = 0; j < order.size(); ++j) {
        const unsigned long long* r = &rec[3 * order[j]];
        int s, a, l;
        amp::del_key_split(r[0], c->Lpad, s, a, l);
        if (sample) sample[j] = s;
        if (anchor) anchor[j] = a;
        if (len) len[j] = l;
        if (count) count[j] = (int32_t)(r[1] & 0xFFFFFFFFULL);
        if (rev) rev[j] = (int32_t)(r[1] >> 32);
        if (qsum) qsum[j] = (int64_t)r[2];
    }
    return AMP_OK;
}

int amp_dels_merge(amp_ctx* c, int64_t n, const int32_t* sample, const int32_t* anchor, const int32_t* len, const int32_t* count,
                   const int32_t* rev, const int64_t* qsum) {
    if (int rc = dels_check(c, "amp_dels_merge")) return rc;
    if (n < 0 || (n > 0 && (!sample || !anchor || !len || !count || !rev || !qsum))) return fail(AMP_ERR_ARG, "amp_dels_merge: bad argument");
    if (n == 0) return AMP_OK;
    std::vector<unsigned long long> in(3 * (size_t)n);
    for (int64_t k = 0; k < n; ++k) {
        if (sample[k] < 0 || sample[k] >= c->cfg.n_samples || anchor[k] < 0 || anchor[k] >= c->cfg.ref_len || len[k] < 1 || count[k] < 0 ||
            rev[k] < 0 || rev[k] > count[k] || qsum[k] < 0)
            return fail(AMP_ERR_ARG, "amp_dels_merge: allele out of range");
        in[3 * k] = amp::del_key(sample[k] * c->Lpad + anchor[k], len[k]);
        in[3 * k + 1] = (unsigned long long)(unsigned int)count[k] | ((unsigned long long)(unsigned int)rev[k] << 32);
        in[3 * k + 2] = (unsigned long long)qsum[k];
    }
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    if (int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n * 24 + 64)) return rc;
    CK(cudaMemcpy(c->d_xbuf, in.data(), (size_t)n * 24, cudaMemcpyHostToDevice));
    amp_dels_merge_kernel<<<(unsigned)std::min<long long>((n + 127) / 128, (long long)c->sm_count * 4), 128>>>(c->dels, (unsigned long long)n,
                                                                                                            (const unsigned long long*)c->d_xbuf);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return AMP_OK;
}

int amp_call_ivar_dels(amp_ctx* c, const amp_ivar_params* p, int32_t* mq, double* pval) {
    if (int rc = dels_check(c, "amp_call_ivar_dels")) return rc;
    if (!p) return fail(AMP_ERR_ARG, "amp_call_ivar_dels: null argument");
    if (!c->d_call) return fail(AMP_ERR_STATE, "amp_call_ivar_dels: amp_call / amp_call_device has not been called");
    std::vector<unsigned long long> rec, order;
    if (int rc = dels_download(c, rec, order)) return rc;
    const unsigned long long n = order.size();
    c->last_launches = 0;
    if (n == 0) return AMP_OK;
    if (int rc = dev_grow(&c->d_dels_out, &c->dels_out_words, (size_t)n * 2)) return rc;
    amp::IvarDelParams P{};
    P.L = c->cfg.ref_len; P.Lpad = c->Lpad; P.dels = c->dels; P.n = n;
    P.depth = (const int*)(c->d_call + c->o_depth);
    P.min_depth = p->min_depth; P.min_freq = p->min_freq;
    P.pval = (double*)c->d_dels_out; P.mq = (int*)(c->d_dels_out + n);
    amp_ivar_dels_kernel<<<(unsigned)((n + 255) / 256), 256>>>(P);
    CK(cudaGetLastError());
    c->last_launches = 1;
    std::vector<int> h_mq(n); std::vector<double> h_pv(n);
    CK(cudaMemcpy(h_pv.data(), P.pval, n * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_mq.data(), P.mq, n * 4, cudaMemcpyDeviceToHost));
    for (unsigned long long j = 0; j < n; ++j) {
        if (mq) mq[j] = h_mq[order[j]];
        if (pval) pval[j] = h_pv[order[j]];
    }
    return AMP_OK;
}

int64_t amp_dels_slot_bytes(int64_t cap_entries) {
    if (cap_entries < 0) return -1;
    return 8 + 8 * AMP_XD_WORDS * cap_entries;
}
int amp_dels_pack_device(amp_ctx* c, void* dev_slot, int64_t cap_entries, void* stream) {
    if (int rc = dels_check(c, "amp_dels_pack_device")) return rc;
    if (!dev_slot || cap_entries < 0) return fail(AMP_ERR_ARG, "amp_dels_pack_device: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    amp_dels_pack_kernel<<<c->sm_count, 256, 0, (cudaStream_t)stream>>>(c->dels, (unsigned long long*)dev_slot, (unsigned long long)cap_entries);
    CK(cudaGetLastError());
    return AMP_OK;
}
int amp_dels_merge_packed(amp_ctx* c, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries, void* stream) {
    if (int rc = dels_check(c, "amp_dels_merge_packed")) return rc;
    if (!dev_slots || n_ranks < 1 || cap_entries < 0) return fail(AMP_ERR_ARG, "amp_dels_merge_packed: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    dim3 grid((unsigned)c->sm_count, (unsigned)n_ranks);
    amp_dels_merge_packed_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(c->dels, (const unsigned long long*)dev_slots,
                                                                        (unsigned long long)amp_dels_slot_bytes(cap_entries) / 8, my_rank);
    CK(cudaGetLastError());
    return AMP_OK;
}

// The blocks of a byte stream that is already in device memory (readable up to d_in + n_bytes + 8): deflate + pack kernels, then the
// BGZF blocks and the EOF block to the host.  Returns the bytes written to out or a negative error code.
static int64_t deflate_device(amp_ctx* c, const uint8_t* d_in, int64_t n_bytes, const int64_t* bstart, int64_t n_blocks, uint8_t* out, int64_t out_cap,
                              cudaStream_t st) {
    static const uint8_t eof[28] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (bstart[0] != 0 || bstart[n_blocks] != n_bytes) return fail(AMP_ERR_ARG, "BGZF deflate: the block table does not cover the data");
    for (int64_t k = 0; k < n_blocks; ++k)
        if (bstart[k + 1] < bstart[k] || bstart[k + 1] - bstart[k] > AMPD_MAXBLOCK) return fail(AMP_ERR_ARG, "BGZF deflate: a block is longer than 0xff00 bytes");
    if (n_blocks == 0) { if (out_cap < 28) return fail(AMP_ERR_ARG, "BGZF deflate: output buffer too small"); memcpy(out, eof, 28); return 28; }
    auto& d = c->defl;
    int rc;
    if ((rc = dev_grow(&d.slots, &d.cap_slots, (size_t)n_blocks * AMPD_SLOT))) return rc;
    if ((rc = dev_grow(&d.bstart, &d.cap_bstart, (size_t)n_blocks + 1))) return rc;
    if ((rc = dev_grow(&d.off, &d.cap_off, (size_t)n_blocks + 1))) return rc;
    if ((rc = dev_grow(&d.clen, &d.cap_clen, (size_t)n_blocks))) return rc;
    if ((rc = dev_grow(&d.crc, &d.cap_crc, (size_t)n_blocks))) return rc;
    if (!d.ctr) CK(cudaMalloc((void**)&d.ctr, 16));
    const size_t smem = ((sizeof(amp::DeflateTables) + 15) & ~(size_t)15) + (size_t)AMPD_WARPS * sizeof(amp::DeflateMem);
    if (!d.attr) { CK(cudaFuncSetAttribute(amp_bgzf_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); d.attr = true; }
    CK(cudaMemcpyAsync(d.bstart, bstart, ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d.ctr, 0, 16, st));
    const int grid = (int)std::min<int64_t>((n_blocks + AMPD_WARPS - 1) / AMPD_WARPS, (int64_t)c->sm_count);
    if ((rc = dev_grow(&d.toks, &d.cap_toks, (size_t)grid * AMPD_WARPS * AMPD_SCRATCH))) return rc;
    amp_bgzf_deflate_kernel<<<grid, AMPD_WARPS * 32, smem, st>>>(d_in, d.bstart, n_blocks, d.slots, d.clen, d.crc, d.ctr, d.toks);
    CK(cudaGetLastError());
    std::vector<uint32_t> clen((size_t)n_blocks);
    CK(cudaMemcpyAsync(clen.data(), d.clen, (size_t)n_blocks * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::vector<long long> off((size_t)n_blocks + 1);
    long long total = 0;
    for (int64_t k = 0; k < n_blocks; ++k) {
        off[(size_t)k] = total;
        total += 26 + (clen[(size_t)k] == 0xFFFFFFFFu ? (bstart[k + 1] - bstart[k]) + 5 : (long long)clen[(size_t)k]);
    }
    off[(size_t)n_blocks] = total;
    if (total + 28 > out_cap) return fail(AMP_ERR_ARG, "BGZF deflate: output buffer too small");
    if ((rc = dev_grow(&d.out, &d.cap_out, (size_t)total + 64))) return rc;
    CK(cudaMemcpyAsync(d.off, off.data(), ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, st));
    amp_bgzf_pack_kernel<<<(unsigned)((n_blocks + 7) / 8), 256, 0, st>>>(d_in, d.bstart, n_blocks, d.slots, d.clen, d.crc, d.off, d.out);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d.out, (size_t)total, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    memcpy(out + total, eof, 28);
    return total + 28;
}

// BGZF-compress host data on the device: in[bstart[k], bstart[k + 1]) becomes block k (each at most 0xff00 bytes; the caller cuts
// at record boundaries the way htslib does), then the EOF block.  Returns the bytes written to out, or a negative error code.
int64_t amp_bgzf_deflate_host(amp_ctx* c, const uint8_t* in, int64_t n_bytes, const int64_t* bstart, int64_t n_blocks, uint8_t* out, int64_t out_cap) {
    if (!c || !in || !bstart || !out || n_bytes < 0 || n_blocks < 0) return fail(AMP_ERR_ARG, "amp_bgzf_deflate_host: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    auto& d = c->defl;
    if (!d.stream) CK(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    int rc;
    if ((rc = dev_grow(&d.in, &d.cap_in, (size_t)n_bytes + 64))) return rc;
    CK(cudaMemcpyAsync(d.in, in, (size_t)n_bytes, cudaMemcpyHostToDevice, d.stream));
    CK(cudaMemsetAsync(d.in + n_bytes, 0, 64, d.stream));
    return deflate_device(c, d.in, n_bytes, bstart, n_blocks, out, out_cap, d.stream);
}

// The trimmed BAM file of the batch amp_bam_decode_host decoded and amp_process_decoded trimmed, built entirely on the device: the
// reads that pass the write gate (AmpliPy.py:910), their records rebuilt with the new pos / bin / n_cigar / CIGAR in the inflated
// input stream that is still in HBM, cut into BGZF blocks at record boundaries (as htslib's bam_write1 does), compressed, and copied to
// the host once.  header = the BAM header (magic, text, references) the file starts with.
int64_t amp_decoded_write_bam(amp_ctx* c, const uint8_t* header, int64_t header_bytes, uint8_t* out, int64_t out_cap, int64_t* n_records) {
    if (!c || !header || !out || header_bytes < 12) return fail(AMP_ERR_ARG, "amp_decoded_write_bam: bad argument");
    auto& d = c->dec;
    if (!d.valid || !d.trimmed) return fail(AMP_ERR_STATE, "amp_decoded_write_bam: no trimmed batch (amp_bam_decode_host + amp_process_decoded with AMP_MODE_TRIM first)");
    CK(cudaSetDevice(c->cfg.device));
    if (!c->defl.stream) CK(cudaStreamCreateWithFlags(&c->defl.stream, cudaStreamNonBlocking));
    cudaStream_t st = c->defl.stream;
    const long long n = d.n_reads;
    int rc;
    if ((rc = dev_grow(&d.w_sizes, &d.cap_wsizes, (size_t)n + 1))) return rc;
    if ((rc = dev_grow(&d.w_off, &d.cap_woff, (size_t)n + 2))) return rc;
    std::vector<unsigned long long> off((size_t)n + 1, 0ULL);
    if (n) {
        amp_bam_newsize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d.raw, d.rec_off, n, d.o_ncig, d.o_flags, d.w_sizes);
        CK(cudaGetLastError());
        amp_scan_sizes_kernel<<<1, 1024, 0, st>>>(d.w_sizes, n, d.w_off);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(off.data(), d.w_off, ((size_t)n + 1) * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    const long long total = header_bytes + (long long)off[(size_t)n];
    // block starts: htslib's layout (whole records per block, up to 0xff00 bytes; the header may share the first block)
    std::vector<int64_t> bstart;
    long long kept = 0;
    {
        const long long BS = AMPD_MAXBLOCK;
        long long cur = 0, prev = 0;
        auto unit = [&](long long end) {                        // a unit [prev, end) joins the open block or starts the next one
            if (end - cur > BS) {
                if (prev > cur) { bstart.push_back(cur); cur = prev; }
                while (end - cur > BS) { bstart.push_back(cur); cur += BS; }
            }
            prev = end;
        };
        unit(header_bytes);
        for (long long i = 0; i < n; ++i) {
            if (off[(size_t)i + 1] == off[(size_t)i]) continue;
            ++kept;
            unit(header_bytes + (long long)off[(size_t)i + 1]);
        }
        if (total > cur) bstart.push_back(cur);
        bstart.push_back(total);
    }
    if (n_records) *n_records = kept;
    if ((rc = dev_grow(&d.w_stream, &d.cap_wstream, (size_t)total + 64))) return rc;
    CK(cudaMemcpyAsync(d.w_stream, header, (size_t)header_bytes, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d.w_stream + total, 0, 64, st));
    if (n) {
        amp_bam_rewrite_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(d.raw, d.rec_off, n, d.cig_off, d.o_pos, d.o_ncig, d.o_cigar, d.w_off, d.w_stream + header_bytes);
        CK(cudaGetLastError());
    }
    return deflate_device(c, d.w_stream, total, bstart.data(), (int64_t)bstart.size() - 1, out, out_cap, st);
}

int amp_host_alloc(void** p, int64_t bytes) {
    if (!p || bytes < 0) return fail(AMP_ERR_ARG, "amp_host_alloc: bad argument");
    CK(cudaHostAlloc(p, (size_t)std::max<int64_t>(bytes, 16), cudaHostAllocDefault));
    return AMP_OK;
}
int amp_host_free(void* p) {
    if (p) CK(cudaFreeHost(p));
    return AMP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// deep-sample mode (SURVEY.md 8e): NCCL sum of the count matrices + packed insertion-table exchange
// ---------------------------------------------------------------------------------------------------
namespace {
struct NcclId { char internal[128]; };
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
// NCCL is resolved at run time (the library already mapped by the host process, e.g. the one PyTorch ships, else the
// system's): the C ABI keeps no link-time dependency on it
NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.handle ? &api : nullptr;
    tried = true;
    const char* names[] = {getenv("AMP_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* nm : names) if (nm && !h) h = dlopen(nm, RTLD_NOW | RTLD_NOLOAD);
    for (const char* nm : names) if (nm && !h) h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (!h) return nullptr;
    api.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    api.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
    api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.AllGather) return nullptr;
    api.handle = h;
    return &api;
}
int nccl_fail(NcclApi* a, int rc, const char* what) {
    return fail(AMP_ERR_CUDA, what, a && a->GetErrorString ? a->GetErrorString(rc) : "NCCL error");
}
#define NCCL_OR_FAIL(a) NcclApi* a = nccl_api(); if (!a) return fail(AMP_ERR_STATE, "NCCL library not found (libnccl.so.2; set AMP_NCCL_LIB)")
}  // namespace

extern "C" {

int amp_nccl_unique_id(uint8_t* id128) {
    if (!id128) return fail(AMP_ERR_ARG, "amp_nccl_unique_id: null argument");
    NCCL_OR_FAIL(a);
    NcclId id;
    const int rc = a->GetUniqueId(&id);
    if (rc) return nccl_fail(a, rc, "ncclGetUniqueId");
    memcpy(id128, id.internal, 128);
    return AMP_OK;
}
int amp_nccl_comm_init(int device, int n_ranks, int rank, const uint8_t* id128, void** comm) {
    if (!id128 || !comm || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(AMP_ERR_ARG, "amp_nccl_comm_init: bad argument");
    NCCL_OR_FAIL(a);
    CK(cudaSetDevice(device));
    NcclId id;
    memcpy(id.internal, id128, 128);
    const int rc = a->CommInitRank(comm, n_ranks, id, rank);
    if (rc) return nccl_fail(a, rc, "ncclCommInitRank");
    return AMP_OK;
}
int amp_nccl_comm_destroy(void* comm) {
    if (!comm) return AMP_OK;
    NCCL_OR_FAIL(a);
    const int rc = a->CommDestroy(comm);
    if (rc) return nccl_fail(a, rc, "ncclCommDestroy");
    return AMP_OK;
}
int amp_nccl_allgather(void* comm, const void* dev_send, void* dev_recv, int64_t bytes_per_rank, void* stream) {
    if (!comm || !dev_send || !dev_recv || bytes_per_rank < 0) return fail(AMP_ERR_ARG, "amp_nccl_allgather: bad argument");
    NCCL_OR_FAIL(a);
    const int rc = a->AllGather(dev_send, dev_recv, (size_t)bytes_per_rank, /*ncclUint8*/ 1, comm, (cudaStream_t)stream);
    if (rc) return nccl_fail(a, rc, "ncclAllGather");
    return AMP_OK;
}

// one ncclAllReduce(sum, int32) over the whole [n_samples][6][lpad] block, in place, asynchronous on `stream`
int amp_allreduce_counts(amp_ctx* c, void* comm, void* stream) {
    if (!c || !comm) return fail(AMP_ERR_ARG, "amp_allreduce_counts: null argument");
    if (c->d_rev) return fail(AMP_ERR_STATE, "amp_allreduce_counts: the context has the strand / quality sums (amp_allreduce_qstats carries them)");
    NCCL_OR_FAIL(a);
    CK(cudaSetDevice(c->cfg.device));
    const size_t n = (size_t)c->cfg.n_samples * AMP_NCH * (size_t)c->Lpad;
    const int rc = a->AllReduce(c->d_counts, c->d_counts, n, /*ncclInt32*/ 2, /*ncclSum*/ 0, comm, (cudaStream_t)stream);
    if (rc) return nccl_fail(a, rc, "ncclAllReduce");
    return AMP_OK;
}

int64_t amp_ins_slot_bytes(int64_t cap_entries, int64_t cap_arena_bytes) {
    if (cap_entries < 0 || cap_arena_bytes < 0) return -1;
    return 16 + 16 * cap_entries + ((cap_arena_bytes + 7) & ~(int64_t)7);
}
int amp_ins_pack_device(amp_ctx* c, void* dev_slot, int64_t cap_entries, int64_t cap_arena_bytes, void* stream) {
    if (!c || !dev_slot || cap_entries < 0 || cap_arena_bytes < 0) return fail(AMP_ERR_ARG, "amp_ins_pack_device: bad argument");
    if (c->d_rev) return fail(AMP_ERR_STATE, "amp_ins_pack_device: the context has the strand / quality sums (amp_ins_pack_qstats_device carries them)");
    CK(cudaSetDevice(c->cfg.device));
    amp_ins_pack_kernel<<<c->sm_count * 2, 512, 0, (cudaStream_t)stream>>>(c->tab, (unsigned long long*)dev_slot, (unsigned long long)cap_entries,
                                                                          (unsigned long long)((cap_arena_bytes + 7) / 8));
    CK(cudaGetLastError());
    return AMP_OK;
}
int amp_ins_merge_packed(amp_ctx* c, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries, int64_t cap_arena_bytes,
                         void* stream) {
    if (!c || !dev_slots || n_ranks < 1 || cap_entries < 0 || cap_arena_bytes < 0) return fail(AMP_ERR_ARG, "amp_ins_merge_packed: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    const unsigned long long slot_words = (unsigned long long)amp_ins_slot_bytes(cap_entries, cap_arena_bytes) / 8;
    dim3 grid((unsigned)c->sm_count, (unsigned)n_ranks);
    amp_ins_merge_packed_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(c->tab, (const unsigned long long*)dev_slots, slot_words,
                                                                       (unsigned long long)cap_entries, my_rank);
    CK(cudaGetLastError());
    return AMP_OK;
}

// The exchange of a context with the strand / quality sums (amp_qstats_enable): the entry points above refuse it, these carry the
// sums.  Three ncclAllReduce(sum) over [n_samples][6][lpad] blocks, in place, asynchronous on `stream`: counts and rev (int32), qsum
// (uint64).
int amp_allreduce_qstats(amp_ctx* c, void* comm, void* stream) {
    if (!c || !comm) return fail(AMP_ERR_ARG, "amp_allreduce_qstats: null argument");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_allreduce_qstats: amp_qstats_enable has not been called");
    NCCL_OR_FAIL(a);
    CK(cudaSetDevice(c->cfg.device));
    const size_t n = (size_t)c->cfg.n_samples * AMP_NCH * (size_t)c->Lpad;
    int rc = a->AllReduce(c->d_counts, c->d_counts, n, /*ncclInt32*/ 2, /*ncclSum*/ 0, comm, (cudaStream_t)stream);
    if (!rc) rc = a->AllReduce(c->d_rev, c->d_rev, n, /*ncclInt32*/ 2, /*ncclSum*/ 0, comm, (cudaStream_t)stream);
    if (!rc) rc = a->AllReduce(c->d_qsum, c->d_qsum, n, /*ncclUint64*/ 5, /*ncclSum*/ 0, comm, (cudaStream_t)stream);
    if (rc) return nccl_fail(a, rc, "ncclAllReduce");
    return AMP_OK;
}

int64_t amp_ins_slot_bytes_qstats(int64_t cap_entries, int64_t cap_arena_bytes) {
    if (cap_entries < 0 || cap_arena_bytes < 0) return -1;
    return 16 + 8 * AMP_XQ_WORDS * cap_entries + ((cap_arena_bytes + 7) & ~(int64_t)7);
}
int amp_ins_pack_qstats_device(amp_ctx* c, void* dev_slot, int64_t cap_entries, int64_t cap_arena_bytes, void* stream) {
    if (!c || !dev_slot || cap_entries < 0 || cap_arena_bytes < 0) return fail(AMP_ERR_ARG, "amp_ins_pack_qstats_device: bad argument");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_ins_pack_qstats_device: amp_qstats_enable has not been called");
    CK(cudaSetDevice(c->cfg.device));
    const amp::QStatsSlots q{c->d_ins_rev, c->d_ins_qsum, c->d_ins_head};
    amp_ins_pack_qstats_kernel<<<c->sm_count * 2, 512, 0, (cudaStream_t)stream>>>(c->tab, q, (unsigned long long*)dev_slot,
                                                                                 (unsigned long long)cap_entries,
                                                                                 (unsigned long long)((cap_arena_bytes + 7) / 8));
    CK(cudaGetLastError());
    return AMP_OK;
}
int amp_ins_merge_packed_qstats(amp_ctx* c, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries, int64_t cap_arena_bytes,
                                void* stream) {
    if (!c || !dev_slots || n_ranks < 1 || cap_entries < 0 || cap_arena_bytes < 0)
        return fail(AMP_ERR_ARG, "amp_ins_merge_packed_qstats: bad argument");
    if (!c->d_rev) return fail(AMP_ERR_STATE, "amp_ins_merge_packed_qstats: amp_qstats_enable has not been called");
    CK(cudaSetDevice(c->cfg.device));
    const amp::QStatsSlots q{c->d_ins_rev, c->d_ins_qsum, c->d_ins_head};
    const unsigned long long slot_words = (unsigned long long)amp_ins_slot_bytes_qstats(cap_entries, cap_arena_bytes) / 8;
    dim3 grid((unsigned)c->sm_count, (unsigned)n_ranks);
    amp_ins_merge_packed_qstats_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(c->tab, q, (const unsigned long long*)dev_slots, slot_words,
                                                                              (unsigned long long)cap_entries, my_rank);
    CK(cudaGetLastError());
    return AMP_OK;
}

// Allocate what amp_process_device would otherwise allocate lazily (long-CIGAR scratch rows, overflow of the per-CTA lists)
// for batches of up to max_reads reads / max_cigar_ops CIGAR ops, so that no later call allocates or synchronises.
int amp_reserve(amp_ctx* c, int64_t max_reads, int64_t max_cigar_ops) {
    if (!c || max_reads < 0 || max_cigar_ops < 0) return fail(AMP_ERR_ARG, "amp_reserve: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t need_s = 2 * ((size_t)max_cigar_ops + 3 * (size_t)max_reads);
    if (need_s > c->scratch_words) {
        if (c->d_scratch) CK(cudaFree(c->d_scratch));
        c->d_scratch = nullptr; c->scratch_words = 0;
        CK(cudaMalloc((void**)&c->d_scratch, need_s * 4));
        c->scratch_words = need_s;
    }
    const size_t need_g = glist_words_for(c, max_reads);
    if (need_g > c->glist_words) {
        if (c->d_glist) CK(cudaFree(c->d_glist));
        c->d_glist = nullptr; c->glist_words = 0;
        CK(cudaMalloc((void**)&c->d_glist, need_g * 4));
        c->glist_words = need_g;
    }
    return AMP_OK;
}

// device-to-device copy of the count matrices into a caller-owned buffer of the same shape (asynchronous on `stream`)
int amp_counts_copy_device(amp_ctx* c, int32_t* dev_dst, void* stream) {
    if (!c || !dev_dst) return fail(AMP_ERR_ARG, "amp_counts_copy_device: null argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaMemcpyAsync(dev_dst, c->d_counts, (size_t)c->cfg.n_samples * AMP_NCH * c->Lpad * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return AMP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// BAM on the device: the compressed file crosses PCIe as it is and is decoded in HBM (amp_bgzf.cuh)
// ---------------------------------------------------------------------------------------------------
extern "C" {

int amp_bam_decode_host(amp_ctx* c, const uint8_t* bgzf, int64_t n_bytes, const int64_t* block_off, const uint32_t* block_isize,
                        int64_t n_blocks, int64_t body_off, amp_bam_info* info) {
    if (!c || !bgzf || !block_off || !block_isize || !info || n_bytes < 0 || n_blocks < 0 || body_off < 0)
        return fail(AMP_ERR_ARG, "amp_bam_decode_host: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    auto& d = c->dec;
    d.valid = false; d.trimmed = false;
    if (c->ct.source == 1) c->ct.source = 0;
    cudaStream_t sc = c->chunk[0].stream, sx = c->chunk[1].stream;    // compute / copy
    CK(cudaStreamSynchronize(sc)); CK(cudaStreamSynchronize(sx));
    // host-side tables: block ends, output offsets
    std::vector<long long> in_off((size_t)n_blocks + 1), out_off((size_t)n_blocks + 1);
    long long raw_len = 0;
    for (int64_t k = 0; k < n_blocks; ++k) {
        if (block_off[k] < 0 || block_off[k] + 28 > n_bytes || (k && block_off[k] <= block_off[k - 1])) return fail(AMP_ERR_ARG, "amp_bam_decode_host: bad block table");
        in_off[k] = block_off[k]; out_off[k] = raw_len; raw_len += block_isize[k];
    }
    in_off[n_blocks] = n_bytes; out_off[n_blocks] = raw_len;
    if (body_off > raw_len) return fail(AMP_ERR_ARG, "amp_bam_decode_host: body offset beyond the stream");
    int rc;
    if ((rc = dev_grow(&d.comp, &d.cap_comp, (size_t)n_bytes + 64))) return rc;
    if ((rc = dev_grow(&d.raw, &d.cap_raw, (size_t)raw_len + 64))) return rc;
    if ((size_t)n_blocks + 1 > d.cap_blocks) {
        const size_t want = (size_t)n_blocks + 1 + 256;
        cudaFree(d.in_off); cudaFree(d.out_off); cudaFree(d.out_len); cudaFree(d.tot); cudaFree(d.prefix);
        d.in_off = d.out_off = nullptr; d.out_len = nullptr; d.tot = nullptr; d.prefix = nullptr; d.cap_blocks = 0;
        CK(cudaMalloc((void**)&d.in_off, want * 8)); CK(cudaMalloc((void**)&d.out_off, want * 8)); CK(cudaMalloc((void**)&d.out_len, want * 4));
        CK(cudaMalloc((void**)&d.tot, want * sizeof(amp::BamBlockTotals))); CK(cudaMalloc((void**)&d.prefix, want * 4 * 8));
        d.cap_blocks = want;
    }
    if (!d.ctr) CK(cudaMalloc((void**)&d.ctr, 64));
    for (auto& e : d.ev) if (!e) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (!d.z_attr) {
        CK(cudaFuncSetAttribute(amp_bgzf_inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(AMPZ_WARPS * sizeof(amp::InflateMem))));
        d.z_attr = true;
    }
    CK(cudaMemcpyAsync(d.in_off, in_off.data(), ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, sx));
    CK(cudaMemcpyAsync(d.out_off, out_off.data(), ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, sx));
    CK(cudaMemcpyAsync(d.out_len, block_isize, (size_t)n_blocks * 4, cudaMemcpyHostToDevice, sx));
    CK(cudaMemsetAsync(d.ctr, 0, 64, sx));
    // One piece.  (Pieces > 1: each is inflated as soon as it has landed, by a launch on a stream of its own, the launches side by
    // side.  Measured with four: 8.9 ms against 8.6 ms end to end -- a block's inflate is latency-bound on one warp, so the call
    // ends one block latency after the LAST piece has landed, and the copy is the smaller part.)
    const int pieces = 1;
    c->last_launches = 0;
    for (int pi = 1; pi < pieces; ++pi) if (!d.zs[pi]) CK(cudaStreamCreateWithFlags(&d.zs[pi], cudaStreamNonBlocking));
    for (int pi = 0; pi < pieces; ++pi) {
        const long long k0 = n_blocks * pi / pieces, k1 = n_blocks * (pi + 1) / pieces;
        if (k1 <= k0) continue;
        const long long b0 = in_off[k0], b1 = in_off[k1];
        cudaStream_t ps = pi == 0 ? sc : d.zs[pi];
        CK(cudaMemcpyAsync(d.comp + b0, bgzf + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, sx));
        CK(cudaEventRecord(d.ev[pi], sx));
        CK(cudaStreamWaitEvent(ps, d.ev[pi], 0));
        const long long nb = k1 - k0;
        const int grid = (int)std::min<long long>((nb + AMPZ_WARPS - 1) / AMPZ_WARPS, (long long)c->sm_count * 2);   // (CTAs of 8 warps: the same 8.7 ms end to end -- the time is one block latency, not contention; one CTA of 24 warps per SM: 12.2 ms)
        amp_bgzf_inflate_kernel<<<grid, AMPZ_WARPS * 32, AMPZ_WARPS * sizeof(amp::InflateMem), ps>>>(d.comp, n_bytes, d.in_off, d.out_len, d.out_off, k0, k1, d.raw,
                                                                                                  d.ctr + 2 + pi, d.ctr + 1);
        CK(cudaGetLastError());
        if (pi > 0) { CK(cudaEventRecord(d.ev[4 + pi], ps)); CK(cudaStreamWaitEvent(sc, d.ev[4 + pi], 0)); }
        c->last_launches += 1;
    }
    unsigned long long tot[4] = {0, 0, 0, 0};
    unsigned int zerr = 0;
    if (n_blocks > 0) {
        amp_bam_count_kernel<<<(unsigned)((n_blocks + 127) / 128), 128, 0, sc>>>(d.raw, d.out_off, n_blocks, body_off, d.tot, d.ctr + 1);
        CK(cudaGetLastError());
        amp_bam_scan_kernel<<<1, 1024, 0, sc>>>(d.tot, n_blocks, d.prefix);
        CK(cudaGetLastError());
        c->last_launches += 2;
        const size_t st = (size_t)n_blocks + 1;
        for (int k = 0; k < 4; ++k) CK(cudaMemcpyAsync(&tot[k], d.prefix + k * st + n_blocks, 8, cudaMemcpyDeviceToHost, sc));
        CK(cudaMemcpyAsync(&zerr, d.ctr + 1, 4, cudaMemcpyDeviceToHost, sc));
    }
    CK(cudaStreamSynchronize(sc));
    if (zerr & (AMPZ_E_DATA | AMPZ_E_SIZE)) return fail(AMP_ERR_DATA, "amp_bam_decode_host: corrupt BGZF block");
    if (zerr & AMPZ_E_ALIGN) return fail(AMP_ERR_DATA, "amp_bam_decode_host: a BAM record straddles a BGZF block boundary (not written by htslib?): use the host decoder");
    if (tot[2] >= (1ULL << 32) || tot[3] >= (1ULL << 32) || tot[1] >= (1ULL << 32)) return fail(AMP_ERR_DATA, "amp_bam_decode_host: more than 4 GiB of bases in one batch; split the input");
    const size_t n = (size_t)tot[0];
    if (n + 1 > d.cap_reads) {
        const size_t want = n + 1 + n / 8 + 64;
        void** arrs[] = {(void**)&d.pos, (void**)&d.flag, (void**)&d.tlen, (void**)&d.cig_off, (void**)&d.seq_off, (void**)&d.qual_off,
                         (void**)&d.rec_off, (void**)&d.o_pos, (void**)&d.o_ncig, (void**)&d.o_flags};
        for (void** ap : arrs) { if (*ap) CK(cudaFree(*ap)); *ap = nullptr; CK(cudaMalloc(ap, want * 8)); }
        d.cap_reads = want;
    }
    if ((rc = dev_grow(&d.cigar, &d.cap_cig, (size_t)tot[1] + 8))) return rc;
    if ((rc = dev_grow(&d.seq, &d.cap_seq, (size_t)tot[2] + 64))) return rc;
    if ((rc = dev_grow(&d.qual, &d.cap_qual, (size_t)tot[3] + 64))) return rc;
    if (n_blocks > 0 && n > 0) {
        amp::BamSoa D{d.pos, d.flag, d.tlen, d.cig_off, d.cigar, d.seq_off, d.seq, d.qual_off, d.qual, d.rec_off};
        amp_bam_scatter_kernel<<<(unsigned)((n_blocks * 32 + 255) / 256), 256, 0, sc>>>(d.raw, d.out_off, n_blocks, body_off, d.prefix, D);
        CK(cudaGetLastError());
        c->last_launches += 1;
    } else {
        CK(cudaMemsetAsync(d.cig_off, 0, 4, sc)); CK(cudaMemsetAsync(d.seq_off, 0, 4, sc)); CK(cudaMemsetAsync(d.qual_off, 0, 4, sc));
    }
    d.n_reads = (long long)n; d.sum_cig = (long long)tot[1]; d.sum_seq = (long long)tot[2]; d.sum_qual = (long long)tot[3];
    d.n_blocks = n_blocks; d.raw_len = raw_len; d.valid = true;
    info->n_reads = d.n_reads; info->sum_cigar_ops = d.sum_cig; info->sum_seq_bytes = d.sum_seq; info->sum_qual_bytes = d.sum_qual;
    info->raw_bytes = raw_len;
    return AMP_OK;
}

int amp_process_decoded(amp_ctx* c, int mode, int sample, const amp_trim_out* host_out) {
    if (!c) return fail(AMP_ERR_ARG, "amp_process_decoded: null context");
    auto& d = c->dec;
    if (!d.valid) return fail(AMP_ERR_STATE, "amp_process_decoded: no decoded batch (amp_bam_decode_host first)");
    if (sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_process_decoded: sample out of range");
    if ((mode & AMP_MODE_TRIM) && !has_scheme(c, sample)) return fail(AMP_ERR_ARG, "amp_process_decoded: trimming needs primer tables");
    if (!(mode & (AMP_MODE_TRIM | AMP_MODE_PILEUP))) return fail(AMP_ERR_ARG, "amp_process_decoded: empty mode");
    if (int rc = check_qstats_mode(c, mode, "amp_process_decoded")) return rc;
    CK(cudaSetDevice(c->cfg.device));
    cudaStream_t sc = c->chunk[0].stream;
    const bool trim = mode & AMP_MODE_TRIM;
    const size_t n = (size_t)d.n_reads, orows = (size_t)d.sum_cig + 3 * n;
    int rc;
    if (trim) {
        if ((rc = dev_grow(&d.o_cigar, &d.cap_ocig, orows + 8))) return rc;
        if ((rc = dev_grow(&d.scratch, &d.cap_scratch, 2 * (orows + 8)))) return rc;
    }
    {
        const size_t need = glist_words_for(c, (long long)n);
        if (need > c->glist_words) {
            if (c->d_glist) CK(cudaFree(c->d_glist));
            c->d_glist = nullptr; c->glist_words = 0;
            CK(cudaMalloc((void**)&c->d_glist, need * 4));
            c->glist_words = need;
        }
    }
    c->last_launches = 0;
    amp::BatchPtrs bp{0, (long long)n, d.pos, d.flag, d.tlen, d.cig_off, d.cigar, d.seq_off, d.seq, d.qual_off, d.qual};
    amp::TrimOut to{};
    if (trim) { to.pos = d.o_pos; to.ncig = d.o_ncig; to.flags = d.o_flags; to.cigar = d.o_cigar; }
    if ((rc = launch_process(c, bp, d.sum_cig, 0, d.sum_qual > 0 ? d.sum_qual : 1, mode, sample, to, trim ? d.scratch : nullptr, c->d_glist, sc))) return rc;
    if (trim) d.trimmed = true;
    if (trim && host_out && n) {
        if (host_out->pos) CK(cudaMemcpyAsync(host_out->pos, d.o_pos, n * 4, cudaMemcpyDeviceToHost, sc));
        if (host_out->ncig) CK(cudaMemcpyAsync(host_out->ncig, d.o_ncig, n * 2, cudaMemcpyDeviceToHost, sc));
        if (host_out->flags) CK(cudaMemcpyAsync(host_out->flags, d.o_flags, n, cudaMemcpyDeviceToHost, sc));
        if (host_out->cigar) CK(cudaMemcpyAsync(host_out->cigar, d.o_cigar, orows * 4, cudaMemcpyDeviceToHost, sc));
    }
    CK(cudaStreamSynchronize(sc));
    return AMP_OK;
}

// the decoded batch back on the host (parity tests, the command line's BAM writer): any pointer may be NULL
int amp_decoded_copy_host(amp_ctx* c, const amp_batch_out* h, uint64_t* rec_off) {
    if (!c || !h) return fail(AMP_ERR_ARG, "amp_decoded_copy_host: null argument");
    auto& d = c->dec;
    if (!d.valid) return fail(AMP_ERR_STATE, "amp_decoded_copy_host: no decoded batch");
    CK(cudaSetDevice(c->cfg.device));
    cudaStream_t sc = c->chunk[0].stream;
    const size_t n = (size_t)d.n_reads;
    if (h->pos) CK(cudaMemcpyAsync(h->pos, d.pos, n * 4, cudaMemcpyDeviceToHost, sc));
    if (h->flag) CK(cudaMemcpyAsync(h->flag, d.flag, n * 2, cudaMemcpyDeviceToHost, sc));
    if (h->tlen) CK(cudaMemcpyAsync(h->tlen, d.tlen, n * 4, cudaMemcpyDeviceToHost, sc));
    if (h->cig_off) CK(cudaMemcpyAsync(h->cig_off, d.cig_off, (n + 1) * 4, cudaMemcpyDeviceToHost, sc));
    if (h->seq_off) CK(cudaMemcpyAsync(h->seq_off, d.seq_off, (n + 1) * 4, cudaMemcpyDeviceToHost, sc));
    if (h->qual_off) CK(cudaMemcpyAsync(h->qual_off, d.qual_off, (n + 1) * 4, cudaMemcpyDeviceToHost, sc));
    if (h->cigar && d.sum_cig) CK(cudaMemcpyAsync(h->cigar, d.cigar, (size_t)d.sum_cig * 4, cudaMemcpyDeviceToHost, sc));
    if (h->seq && d.sum_seq) CK(cudaMemcpyAsync(h->seq, d.seq, (size_t)d.sum_seq, cudaMemcpyDeviceToHost, sc));
    if (h->qual && d.sum_qual) CK(cudaMemcpyAsync(h->qual, d.qual, (size_t)d.sum_qual, cudaMemcpyDeviceToHost, sc));
    if (rec_off && n) CK(cudaMemcpyAsync(rec_off, d.rec_off, n * 8, cudaMemcpyDeviceToHost, sc));
    CK(cudaStreamSynchronize(sc));
    return AMP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// heterogeneous plates (SURVEY.md 8f-4): a primer scheme / reference per sample, tables built on the device
// ---------------------------------------------------------------------------------------------------
// find_overlapping_primers (AmpliPy.py:174-209) as its covering-set definition: position p takes the smallest start / largest
// end over the primers with start - offset <= p < end + offset (the offset widens the coverage only); -1 = uncovered
__global__ void amp_primer_tables_kernel(int L, const int32_t* start, const int32_t* end, int n, int offset, int32_t* mn, int32_t* mx) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= L) return;
    int lo = 0x7FFFFFFF, hi = -1;
    for (int k = 0; k < n; ++k) {
        const int s = start[k], e = end[k];
        if (s - offset <= p && p < e + offset) { lo = s < lo ? s : lo; hi = e > hi ? e : hi; }
    }
    mn[p] = hi < 0 ? -1 : lo; mx[p] = hi;
}

extern "C" {

int amp_set_scheme(amp_ctx* c, int sample, int32_t ref_len, const int32_t* primer_start, const int32_t* primer_end, int32_t n_primers,
                   int32_t offset) {
    if (!c || sample < 0 || sample >= c->cfg.n_samples || ref_len < 1 || ref_len > c->cfg.ref_len || n_primers < 0 || offset < 0 ||
        (n_primers && (!primer_start || !primer_end)))
        return fail(AMP_ERR_ARG, "amp_set_scheme: bad argument (the sample's reference must not be longer than the context's ref_len)");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    if (c->scheme.size() < (size_t)c->cfg.n_samples) c->scheme.resize((size_t)c->cfg.n_samples);
    auto& sc = c->scheme[sample];
    if (!sc.d_min) { CK(cudaMalloc((void**)&sc.d_min, (size_t)c->cfg.ref_len * 4)); CK(cudaMalloc((void**)&sc.d_max, (size_t)c->cfg.ref_len * 4)); }
    int32_t *d_s = nullptr, *d_e = nullptr;
    int mpl = 0;
    for (int k = 0; k < n_primers; ++k) mpl = std::max(mpl, primer_end[k] - primer_start[k]);
    {
        int rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n_primers * 8 + 64);
        if (rc) return rc;
    }
    d_s = (int32_t*)c->d_xbuf; d_e = d_s + n_primers;
    if (n_primers) {
        CK(cudaMemcpy(d_s, primer_start, (size_t)n_primers * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_e, primer_end, (size_t)n_primers * 4, cudaMemcpyHostToDevice));
    }
    amp_primer_tables_kernel<<<(ref_len + 255) / 256, 256>>>(ref_len, d_s, d_e, n_primers, offset, sc.d_min, sc.d_max);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    sc.L = ref_len; sc.mpl = mpl;
    return AMP_OK;
}

// the tables of a sample's scheme back on the host (tests: the device-side build against find_overlapping_primers)
int amp_get_scheme(amp_ctx* c, int sample, int32_t* min_primer_start, int32_t* max_primer_end, int32_t* max_primer_len) {
    if (!c || sample < 0 || (size_t)sample >= c->scheme.size() || c->scheme[sample].L < 1) return fail(AMP_ERR_ARG, "amp_get_scheme: no scheme for this sample");
    CK(cudaSetDevice(c->cfg.device));
    const auto& sc = c->scheme[sample];
    if (min_primer_start) CK(cudaMemcpy(min_primer_start, sc.d_min, (size_t)sc.L * 4, cudaMemcpyDeviceToHost));
    if (max_primer_end) CK(cudaMemcpy(max_primer_end, sc.d_max, (size_t)sc.L * 4, cudaMemcpyDeviceToHost));
    if (max_primer_len) *max_primer_len = sc.mpl;
    return AMP_OK;
}

// a reference of its own for one sample (at most ref_len characters; positions past its end are called as 'N' with depth 0)
int amp_set_sample_reference(amp_ctx* c, int sample, const char* ref_seq, int32_t len) {
    if (!c || !ref_seq || sample < 0 || sample >= c->cfg.n_samples || len < 1 || len > c->cfg.ref_len) return fail(AMP_ERR_ARG, "amp_set_sample_reference: bad argument");
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaDeviceSynchronize());
    const size_t L = (size_t)c->cfg.ref_len, S = (size_t)c->cfg.n_samples;
    if (!c->ref_per_sample) {
        unsigned char* nr = nullptr;
        CK(cudaMalloc((void**)&nr, S * L + 16));
        CK(cudaMemset(nr, 'N', S * L));
        if (c->d_ref) { for (size_t k = 0; k < S; ++k) CK(cudaMemcpy(nr + k * L, c->d_ref, L, cudaMemcpyDeviceToDevice)); CK(cudaFree(c->d_ref)); }
        c->d_ref = nr; c->ref_per_sample = true;
    }
    CK(cudaMemset(c->d_ref + (size_t)sample * L, 'N', L));
    CK(cudaMemcpy(c->d_ref + (size_t)sample * L, ref_seq, (size_t)len, cudaMemcpyHostToDevice));
    if (c->ref_len_s.size() != S) c->ref_len_s.assign(S, (int)L);
    c->ref_len_s[sample] = len;
    c->an.built = false;
    return AMP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// a batch grouped by contig (amp_contig.cuh, DESIGN.md 3.8): contig k = sample k of the context
// ---------------------------------------------------------------------------------------------------
namespace {

// plan kernel + one copy of its table; P.raw / rec_off / ref_to_sample or P.sample_in set by the caller
int contig_plan(amp_ctx* c, amp::ContigPlanParams P, const amp::BatchPtrs& b, int source, amp_contig_plan* plan) {
    auto& t = c->ct;
    t.source = 0;
    const int S = c->cfg.n_samples;
    if (S > AMP_MAX_CONTIGS) return fail(AMP_ERR_ARG, "amp_contig_plan: more contigs than AMP_MAX_CONTIGS (1024)");
    cudaStream_t sc = c->chunk[0].stream;
    const long long n = b.n, n_tiles = (n + AMP_CT_TILE - 1) / AMP_CT_TILE;
    const size_t words = amp::ct_table_words(S, P.n_refs);
    int rc;
    if ((rc = dev_grow(&t.sid, &t.cap_sid, (size_t)n + 1))) return rc;
    if ((rc = dev_grow(&t.hist, &t.cap_hist, (size_t)n_tiles * S + 1))) return rc;
    if ((rc = dev_grow(&t.table, &t.cap_table, words))) return rc;
    CK(cudaMemsetAsync(t.table, 0, words * 8, sc));
    P.n = n; P.flag = b.flag; P.cig_off = b.cig_off; P.qual_off = b.qual_off; P.S = S;
    P.sid = t.sid; P.tile_hist = t.hist; P.table = t.table;
    c->last_launches = 0;
    if (n_tiles) {
        amp_contig_plan_kernel<<<(unsigned)n_tiles, AMP_CT_THREADS, 0, sc>>>(P);
        CK(cudaGetLastError());
        c->last_launches = 1;
    }
    t.h_table.assign(words, 0ULL);
    CK(cudaMemcpyAsync(t.h_table.data(), t.table, words * 8, cudaMemcpyDeviceToHost, sc));
    CK(cudaStreamSynchronize(sc));
    const unsigned long long* T = t.h_table.data();
    int present = T[0] ? 1 : 0;
    for (int k = 0; k < S; ++k) present += T[AMP_CT_HDR + k] ? 1 : 0;
    plan->n_reads = n; plan->n_no_contig = (int64_t)T[0]; plan->errors = (uint32_t)T[2];
    plan->grouped = (n == 0 || T[1] + 1 == (unsigned long long)present) ? 1 : 0;
    for (int k = 0; k < S; ++k) {
        const unsigned long long cnt = T[AMP_CT_HDR + k];
        if (plan->contig_reads) plan->contig_reads[k] = (int64_t)cnt;
        if (plan->contig_first) plan->contig_first[k] = cnt ? (int64_t)~T[AMP_CT_HDR + 3 * (size_t)S + k] : 0;
        if (plan->contig_cigar_ops) plan->contig_cigar_ops[k] = (int64_t)T[AMP_CT_HDR + (size_t)S + k];
        if (plan->contig_qual_bytes) plan->contig_qual_bytes[k] = (int64_t)T[AMP_CT_HDR + 2 * (size_t)S + k];
    }
    if (plan->ref_reads) for (int r = 0; r < P.n_refs; ++r) plan->ref_reads[r] = (int64_t)T[AMP_CT_HDR + 5 * (size_t)S + r];
    t.b = b; t.sum_cig = (long long)T[3]; t.grouped = plan->grouped != 0;
    t.source = source;
    return AMP_OK;
}

// the permuted copy of the planned batch: one range per contig, in contig order, into t.pos ... t.qual
int contig_permute(amp_ctx* c, cudaStream_t sc) {
    auto& t = c->ct;
    const int S = c->cfg.n_samples;
    const long long n = t.b.n, n_tiles = (n + AMP_CT_TILE - 1) / AMP_CT_TILE;
    const unsigned long long* T = t.h_table.data();
    long long sum_seq = 0, sum_qual = 0, n_in = 0;
    for (int k = 0; k < S; ++k) { n_in += (long long)T[AMP_CT_HDR + k]; sum_qual += (long long)T[AMP_CT_HDR + 2 * (size_t)S + k]; }
    int rc;
    if ((rc = dev_grow(&t.hist_off, &t.cap_hoff, (size_t)n_tiles * S + 1))) return rc;
    if ((rc = dev_grow(&t.perm, &t.cap_perm, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.tsum, &t.cap_tsum, (size_t)n_tiles * 3 + 3))) return rc;
    if ((rc = dev_grow(&t.tbase, &t.cap_tbase, 3 * ((size_t)n_tiles + 1) + 3))) return rc;
    // contig-major prefix sums of the tile histograms: the place of each tile's first read of each contig
    amp::ContigScanParams H{t.hist, (long long)S * n_tiles, n_tiles, (long long)S, 1, t.hist_off};
    amp_contig_scan_kernel<<<dim3(1, 1), AMP_CT_THREADS, 0, sc>>>(H, H, H);
    CK(cudaGetLastError());
    amp::ContigRankParams R{n, S, n_tiles, t.sid, t.hist_off, t.perm};
    amp_contig_rank_kernel<<<(unsigned)n_tiles, AMP_CT_THREADS, 0, sc>>>(R);
    CK(cudaGetLastError());
    // rows of the permuted batch: the seq bytes are not in the plan (they follow from the quality bytes); size them from those
    sum_seq = sum_qual / 2 + n_in;
    const long long pt = (n_in + AMP_CT_TILE - 1) / AMP_CT_TILE;
    if ((rc = dev_grow(&t.pos, &t.cap_pos, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.flag, &t.cap_flag, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.tlen, &t.cap_tlen, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.cig_off, &t.cap_coff, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.seq_off, &t.cap_soff, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.qual_off, &t.cap_qoff, (size_t)n_in + 1))) return rc;
    if ((rc = dev_grow(&t.cigar, &t.cap_cig, (size_t)t.sum_cig + 8))) return rc;
    if ((rc = dev_grow(&t.seq, &t.cap_seq, (size_t)sum_seq + 64))) return rc;          // + the 16-byte reads past the end (DESIGN.md 2)
    if ((rc = dev_grow(&t.qual, &t.cap_qual, (size_t)sum_qual + 64))) return rc;
    amp::ContigGatherParams G{};
    G.n = n_in; G.n_tiles = pt; G.perm = t.perm; G.src = t.b; G.src.first = 0;
    G.pos = t.pos; G.flag = t.flag; G.tlen = t.tlen; G.cig_off = t.cig_off; G.cigar = t.cigar; G.seq_off = t.seq_off; G.seq = t.seq;
    G.qual_off = t.qual_off; G.qual = t.qual; G.tsum = t.tsum; G.tbase = t.tbase;
    if (n_in == 0) {
        CK(cudaMemsetAsync(t.cig_off, 0, 4, sc)); CK(cudaMemsetAsync(t.seq_off, 0, 4, sc)); CK(cudaMemsetAsync(t.qual_off, 0, 4, sc));
        c->last_launches += 2;
        return AMP_OK;
    }
    amp_contig_tilesum_kernel<<<(unsigned)pt, AMP_CT_THREADS, 0, sc>>>(G);
    CK(cudaGetLastError());
    amp::ContigScanParams Q[3];
    for (int ch = 0; ch < 3; ++ch) Q[ch] = amp::ContigScanParams{t.tsum + ch, pt, pt, 3, 0, t.tbase + (size_t)ch * (pt + 1)};
    amp_contig_scan_kernel<<<dim3(1, 3), AMP_CT_THREADS, 0, sc>>>(Q[0], Q[1], Q[2]);
    CK(cudaGetLastError());
    amp_contig_gather_kernel<<<(unsigned)pt, AMP_CT_THREADS, 0, sc>>>(G);
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(t.seq + sum_seq, 0, 64, sc));
    c->last_launches += 5;
    return AMP_OK;
}

}  // namespace

extern "C" {

int amp_contig_plan_decoded(amp_ctx* c, const int32_t* ref_to_sample, int32_t n_refs, amp_contig_plan* plan) {
    if (!c || !plan || n_refs < 0 || (n_refs && !ref_to_sample)) return fail(AMP_ERR_ARG, "amp_contig_plan_decoded: bad argument");
    auto& d = c->dec;
    if (!d.valid) return fail(AMP_ERR_STATE, "amp_contig_plan_decoded: no decoded batch (amp_bam_decode_host first)");
    CK(cudaSetDevice(c->cfg.device));
    int rc;
    if ((rc = dev_grow(&c->d_xbuf, &c->xbuf_bytes, (size_t)n_refs * 4 + 64))) return rc;
    int* d_map = (int*)c->d_xbuf;
    if (n_refs) CK(cudaMemcpyAsync(d_map, ref_to_sample, (size_t)n_refs * 4, cudaMemcpyHostToDevice, c->chunk[0].stream));
    amp::ContigPlanParams P{};
    P.raw = d.raw; P.rec_off = d.rec_off; P.ref_to_sample = d_map; P.n_refs = n_refs;
    amp::BatchPtrs b{0, d.n_reads, d.pos, d.flag, d.tlen, d.cig_off, d.cigar, d.seq_off, d.seq, d.qual_off, d.qual};
    return contig_plan(c, P, b, 1, plan);
}

int amp_contig_plan_device(amp_ctx* c, const amp_batch* b, const int32_t* dev_sample_of_read, amp_contig_plan* plan) {
    if (!c || !b || !plan || (b->n_reads && !dev_sample_of_read) || b->first != 0 || b->n_reads < 0)
        return fail(AMP_ERR_ARG, "amp_contig_plan_device: bad argument (the batch must start at read 0)");
    CK(cudaSetDevice(c->cfg.device));
    amp::ContigPlanParams P{};
    P.sample_in = dev_sample_of_read;
    amp::BatchPtrs bp{0, b->n_reads, b->pos, b->flag, b->tlen, b->cig_off, b->cigar, b->seq_off, b->seq, b->qual_off, b->qual};
    if (plan->ref_reads) return fail(AMP_ERR_ARG, "amp_contig_plan_device: ref_reads is for the decoded plan");
    return contig_plan(c, P, bp, 2, plan);
}

int amp_process_contigs(amp_ctx* c, int mode, const amp_trim_out* dev_out, const amp_trim_out* host_out) {
    if (!c) return fail(AMP_ERR_ARG, "amp_process_contigs: null context");
    auto& t = c->ct;
    auto& d = c->dec;
    if (!t.source || (t.source == 1 && !d.valid)) return fail(AMP_ERR_STATE, "amp_process_contigs: no planned batch (amp_contig_plan_* first)");
    const int S = c->cfg.n_samples;
    const unsigned long long* T = t.h_table.data();
    if (T[2]) return fail(AMP_ERR_DATA, "amp_process_contigs: the plan found reads without a valid contig (amp_contig_plan.errors)");
    if (!(mode & (AMP_MODE_TRIM | AMP_MODE_PILEUP))) return fail(AMP_ERR_ARG, "amp_process_contigs: empty mode");
    if (int rc = check_qstats_mode(c, mode, "amp_process_contigs")) return rc;
    const bool trim = mode & AMP_MODE_TRIM;
    if (t.source == 1 && dev_out) return fail(AMP_ERR_ARG, "amp_process_contigs: the decoded batch keeps its trim outputs in the context (dev_out must be NULL)");
    if (t.source == 2 && trim && !dev_out) return fail(AMP_ERR_ARG, "amp_process_contigs: trimming a device batch needs dev_out");
    for (int k = 0; k < S && trim; ++k)
        if (T[AMP_CT_HDR + k] && !has_scheme(c, k)) return fail(AMP_ERR_ARG, "amp_process_contigs: trimming needs a scheme for every contig with reads");
    CK(cudaSetDevice(c->cfg.device));
    cudaStream_t sc = c->chunk[0].stream;
    const long long n = t.b.n;
    const size_t orows = (size_t)t.sum_cig + 3 * (size_t)n;
    int rc;
    amp::TrimOut out{};
    if (trim && t.source == 1) {
        if ((rc = dev_grow(&d.o_cigar, &d.cap_ocig, orows + 8))) return rc;
        out.pos = d.o_pos; out.ncig = d.o_ncig; out.flags = d.o_flags; out.cigar = d.o_cigar;
    } else if (trim) {
        out.pos = dev_out->pos; out.ncig = dev_out->ncig; out.flags = dev_out->flags; out.cigar = dev_out->cigar;
    }
    if (trim && (rc = dev_grow(&t.scratch, &t.cap_scratch, 2 * (orows + 8)))) return rc;
    {
        const size_t need = glist_words_for(c, n);
        if (need > c->glist_words) {
            CK(cudaStreamSynchronize(sc));
            if (c->d_glist) CK(cudaFree(c->d_glist));
            c->d_glist = nullptr; c->glist_words = 0;
            CK(cudaMalloc((void**)&c->d_glist, need * 4));
            c->glist_words = need;
        }
    }
    c->last_launches = 0;
    if (t.grouped) {
        // one launch per contig over its own range of the batch; scratch rows are addressed like the output rows, from the range start
        for (int k = 0; k < S; ++k) {
            const long long cnt = (long long)T[AMP_CT_HDR + k];
            if (!cnt) continue;
            const long long first = (long long)~T[AMP_CT_HDR + 3 * (size_t)S + k], cfirst = (long long)T[AMP_CT_HDR + 4 * (size_t)S + k];
            amp::BatchPtrs bk = t.b;
            bk.first = first; bk.n = cnt;
            const long long scig = (long long)T[AMP_CT_HDR + (size_t)S + k], squal = (long long)T[AMP_CT_HDR + 2 * (size_t)S + k];
            if ((rc = launch_process(c, bk, scig, 0, squal > 0 ? squal : 1, mode, k, out, trim ? t.scratch - (cfirst + 3 * first) : nullptr,
                                     c->d_glist, sc))) return rc;
        }
    } else {
        if ((rc = contig_permute(c, sc))) return rc;
        long long n_in = 0;
        for (int k = 0; k < S; ++k) n_in += (long long)T[AMP_CT_HDR + k];
        amp::TrimOut po{};
        if (trim) {
            if ((rc = dev_grow(&t.o_pos, &t.cap_opos, (size_t)n_in + 1))) return rc;
            if ((rc = dev_grow(&t.o_ncig, &t.cap_oncig, (size_t)n_in + 1))) return rc;
            if ((rc = dev_grow(&t.o_flags, &t.cap_oflags, (size_t)n_in + 1))) return rc;
            if ((rc = dev_grow(&t.o_cigar, &t.cap_ocig, (size_t)t.sum_cig + 3 * (size_t)n_in + 8))) return rc;
            po.pos = t.o_pos; po.ncig = t.o_ncig; po.flags = t.o_flags; po.cigar = t.o_cigar;
        }
        const amp::BatchPtrs pb{0, n_in, t.pos, t.flag, t.tlen, t.cig_off, t.cigar, t.seq_off, t.b.seq ? t.seq : nullptr, t.qual_off, t.qual};
        long long first = 0, cfirst = 0;
        for (int k = 0; k < S; ++k) {
            const long long cnt = (long long)T[AMP_CT_HDR + k];
            const long long scig = (long long)T[AMP_CT_HDR + (size_t)S + k], squal = (long long)T[AMP_CT_HDR + 2 * (size_t)S + k];
            if (cnt) {
                amp::BatchPtrs bk = pb;
                bk.first = first; bk.n = cnt;
                if ((rc = launch_process(c, bk, scig, 0, squal > 0 ? squal : 1, mode, k, po, trim ? t.scratch - (cfirst + 3 * first) : nullptr,
                                         c->d_glist, sc))) return rc;
            }
            first += cnt; cfirst += scig;
        }
        if (trim && n_in) {
            amp::ContigUnpermuteParams U{n_in, t.perm, t.cig_off, po, t.b.cig_off, out};
            const long long grid = std::min<long long>((n_in + 7) / 8, (long long)c->sm_count * 16);
            amp_contig_unpermute_kernel<<<(unsigned)grid, 256, 0, sc>>>(U);
            CK(cudaGetLastError());
            c->last_launches += 1;
        }
    }
    if (trim && T[0]) {
        amp::ContigSkipParams K{n, t.sid, t.b, out};
        const long long grid = std::min<long long>((n + 255) / 256, (long long)c->sm_count * 8);
        amp_contig_skip_kernel<<<(unsigned)grid, 256, 0, sc>>>(K);
        CK(cudaGetLastError());
        c->last_launches += 1;
    }
    if (trim && t.source == 1) d.trimmed = true;
    if (trim && host_out && n) {
        if (host_out->pos) CK(cudaMemcpyAsync(host_out->pos, out.pos, (size_t)n * 4, cudaMemcpyDeviceToHost, sc));
        if (host_out->ncig) CK(cudaMemcpyAsync(host_out->ncig, out.ncig, (size_t)n * 2, cudaMemcpyDeviceToHost, sc));
        if (host_out->flags) CK(cudaMemcpyAsync(host_out->flags, out.flags, (size_t)n, cudaMemcpyDeviceToHost, sc));
        if (host_out->cigar) CK(cudaMemcpyAsync(host_out->cigar, out.cigar, orows * 4, cudaMemcpyDeviceToHost, sc));
    }
    CK(cudaStreamSynchronize(sc));
    return AMP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// codon annotation of the iVar TSV (amp_annot.cuh, DESIGN.md 3.9)
// ---------------------------------------------------------------------------------------------------
namespace {
int sample_ref_len(const amp_ctx* c, int sample) {
    return c->ref_per_sample && (size_t)sample < c->ref_len_s.size() ? c->ref_len_s[sample] : c->cfg.ref_len;
}
}  // namespace

extern "C" {

int amp_set_features(amp_ctx* c, int sample, int32_t n_features, const int32_t* strand, const int32_t* phase, const int32_t* seg_off,
                     const int32_t* seg_start, const int32_t* seg_end) {
    if (!c || sample < 0 || sample >= c->cfg.n_samples) return fail(AMP_ERR_ARG, "amp_set_features: bad sample");
    if (!c->d_ref) return fail(AMP_ERR_STATE, "amp_set_features: no reference (amp_set_reference / amp_set_sample_reference first)");
    amp::AnnotFeatures f;
    if (!amp::annot_features(sample_ref_len(c, sample), n_features, strand, phase, seg_off, seg_start, seg_end, f))
        return fail(AMP_ERR_ARG, "amp_set_features: bad feature (strand +1 / -1, phase 0..2, at least one segment, 0 <= start < end <= the sample's length)");
    if (c->an.feat.size() < (size_t)c->cfg.n_samples) c->an.feat.resize((size_t)c->cfg.n_samples);
    c->an.feat[sample] = std::move(f);
    c->an.built = false;
    return AMP_OK;
}

int amp_annotate(amp_ctx* c, int64_t* n_entries) {
    if (!c) return fail(AMP_ERR_ARG, "amp_annotate: null context");
    auto& a = c->an;
    bool any = false;
    for (size_t s = 0; s < a.feat.size(); ++s) {
        any |= !a.feat[s].lo.empty();
        for (int e : a.feat[s].hi)
            if (e > sample_ref_len(c, (int)s)) return fail(AMP_ERR_ARG, "amp_annotate: a segment ends past its sample's reference");
    }
    if (!any) return fail(AMP_ERR_STATE, "amp_annotate: no features (amp_set_features first)");
    if (!c->d_ref) return fail(AMP_ERR_STATE, "amp_annotate: no reference");
    CK(cudaSetDevice(c->cfg.device));
    a.built = false;
    const int S = c->cfg.n_samples, L = c->cfg.ref_len;
    const long long SL = (long long)S * L, n_tiles = (SL + AMP_AN_THREADS - 1) / AMP_AN_THREADS;
    std::vector<amp::AnnotFeatures> all(a.feat);
    all.resize((size_t)S);
    amp::AnnotTables T;
    amp::annot_tables(all, T);
    const std::vector<int>* parts[] = {&T.samp_seg, &T.sg_lo, &T.sg_max, &T.sg_key, &T.fs_lo, &T.fs_hi, &T.fs_cum, &T.fs_feat, &T.ft_fs,
                                       &T.ft_len, &T.ft_local, &T.ft_info};
    size_t words = 0;
    for (auto* v : parts) words += v->size();
    std::vector<int> packed;
    packed.reserve(words);
    for (auto* v : parts) packed.insert(packed.end(), v->begin(), v->end());
    int rc;
    if ((rc = dev_grow(&a.tables, &a.cap_tables, words)) || (rc = dev_grow(&a.off, &a.cap_off, (size_t)SL + 1)) ||
        (rc = dev_grow(&a.tsum, &a.cap_tsum, (size_t)n_tiles)) || (rc = dev_grow(&a.tbase, &a.cap_tbase, (size_t)n_tiles + 1)))
        return rc;
    cudaStream_t st = c->chunk[0].stream;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyAsync(a.tables, packed.data(), words * 4, cudaMemcpyHostToDevice, st));
    amp::AnnotParams P{};
    P.L = L; P.n_samples = S; P.ref = c->d_ref; P.ref_stride = c->ref_per_sample ? (long long)L : 0;
    const int** dst[] = {&P.samp_seg, &P.sg_lo, &P.sg_max, &P.sg_key, &P.fs_lo, &P.fs_hi, &P.fs_cum, &P.fs_feat, &P.ft_fs, &P.ft_len,
                         &P.ft_local, &P.ft_info};
    size_t o = 0;
    for (int k = 0; k < 12; ++k) { *dst[k] = a.tables + o; o += parts[k]->size(); }
    P.off = a.off;
    amp_annot_count_kernel<<<(unsigned)n_tiles, AMP_AN_THREADS, 0, st>>>(P, a.tsum);
    CK(cudaGetLastError());
    amp::ContigScanParams H{a.tsum, n_tiles, n_tiles, 1, 0, a.tbase};
    amp_contig_scan_kernel<<<dim3(1, 1), AMP_CT_THREADS, 0, st>>>(H, H, H);
    CK(cudaGetLastError());
    uint32_t total = 0;
    CK(cudaMemcpyAsync(&total, a.tbase + n_tiles, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const size_t E = total;
    if ((rc = dev_grow(&a.e_int, &a.cap_eint, 2 * E + 1)) || (rc = dev_grow(&a.e_chr, &a.cap_echr, 25 * E + 1))) return rc;
    P.e_feat = a.e_int; P.e_pos_aa = a.e_int + E;
    P.e_off = a.e_chr; P.e_codon = a.e_chr + E; P.e_aa = a.e_chr + 19 * E;
    amp_annot_fill_kernel<<<(unsigned)n_tiles, AMP_AN_THREADS, 0, st>>>(P, a.tbase, (unsigned)n_tiles);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    c->last_launches = 3;
    a.n = (long long)E; a.built = true;
    if (n_entries) *n_entries = a.n;
    return AMP_OK;
}

int amp_annot_host(amp_ctx* c, uint32_t* off, int32_t* feat, int32_t* pos_aa, uint8_t* codon_off, char* codons, char* aas) {
    if (!c) return fail(AMP_ERR_ARG, "amp_annot_host: null context");
    if (!c->an.built) return fail(AMP_ERR_STATE, "amp_annot_host: no annotation (amp_annotate first, after the last change of features or reference)");
    CK(cudaSetDevice(c->cfg.device));
    auto& a = c->an;
    const size_t SL = (size_t)c->cfg.n_samples * c->cfg.ref_len, E = (size_t)a.n;
    cudaStream_t st = c->chunk[0].stream;
    if (off) CK(cudaMemcpyAsync(off, a.off, (SL + 1) * 4, cudaMemcpyDeviceToHost, st));
    if (E) {
        if (feat) CK(cudaMemcpyAsync(feat, a.e_int, E * 4, cudaMemcpyDeviceToHost, st));
        if (pos_aa) CK(cudaMemcpyAsync(pos_aa, a.e_int + E, E * 4, cudaMemcpyDeviceToHost, st));
        if (codon_off) CK(cudaMemcpyAsync(codon_off, a.e_chr, E, cudaMemcpyDeviceToHost, st));
        if (codons) CK(cudaMemcpyAsync(codons, a.e_chr + E, E * 18, cudaMemcpyDeviceToHost, st));
        if (aas) CK(cudaMemcpyAsync(aas, a.e_chr + 19 * E, E * 6, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return AMP_OK;
}

}  // extern "C"
