/*
 * amplipy_b200.h -- C ABI of the B200-native trim -> pileup -> call path (libamplipy_b200.so).
 *
 * The reference (Niema-Lab/AmpliPy, /root/reference/AmpliPy.py) has no FFI: its hot path is three
 * Python functions called per read / per position.  Each entry point below states which of them it
 * replaces; INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success or a negative AMP_ERR_* code (message from
 * amp_last_error(), thread-local); nothing throws; all buffers are caller-owned; no torch types.
 * "device" pointers are CUDA device pointers on the context's device; `stream` is a cudaStream_t
 * passed as void* (NULL = default stream).
 *
 * Batch layout (struct-of-arrays, one entry per read unless noted; amplipy_b200/batch.py):
 *   pos i32, flag u16, tlen i32, cig_off u32[N+1], cigar u32[sumC] (BAM: len<<4|op),
 *   seq_off u32[N+1] (bytes), seq u8 (BAM 4-bit, (l_seq+1)/2 bytes per read),
 *   qual_off u32[N+1] (bytes; l_seq = diff), qual u8 (phred).
 *   `seq` and `qual` base addresses must be 16-byte aligned, and device copies of them must be readable up to the
 *   next 16-byte boundary past their last byte (the kernels move them in whole 16-byte pieces).
 * Trim output layout: row i of out_cigar starts at cig_off[i] + 3*i (capacity n_cigar[i] + 3).
 */
#ifndef AMPLIPY_B200_H
#define AMPLIPY_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMP_ABI_VERSION 1

/* error codes */
#define AMP_OK 0
#define AMP_ERR_CUDA (-1)
#define AMP_ERR_ARG (-2)
#define AMP_ERR_NOMEM (-3)
#define AMP_ERR_STATE (-4)
#define AMP_ERR_DATA (-5)     /* malformed input data (message says what) */

/* out_flags bits per read (AmpliPy.py:443-447 return tuple of trim_read + write gate 910 + skip 902) */
#define AMP_FLAG_TRIM_START 1
#define AMP_FLAG_TRIM_END 2
#define AMP_FLAG_TRIM_QUAL 4
#define AMP_FLAG_KEEP 8
#define AMP_FLAG_SKIPPED 16
#define AMP_FLAG_ERROR 32

/* device error word bits (amp_error_flags): inputs for which the reference itself crashes */
#define AMP_DEVERR_COORD 1
#define AMP_DEVERR_BASE 2
#define AMP_DEVERR_INS_END 4
#define AMP_DEVERR_CIGAR 8
#define AMP_DEVERR_TABLE_FULL 16
#define AMP_DEVERR_ARENA_FULL 32
#define AMP_DEVERR_QSTATS_MISS 64   /* strand / quality pass: an insertion allele the pileup did not add (never expected) */
#define AMP_DEVERR_DELS_FULL 128    /* anchored deletion table full (amp_dels_enable); the alleles it could not take are lost */

/* mode bits for amp_process_* */
#define AMP_MODE_TRIM 1      /* trim_read, AmpliPy.py:426-687 (+ gate 902/910) */
#define AMP_MODE_PILEUP 2    /* update_base_counts, AmpliPy.py:690-753 */
#define AMP_MODE_QSTATS 4    /* with AMP_MODE_PILEUP, after amp_qstats_enable: strand / quality sums of the same events */

typedef struct amp_ctx amp_ctx;

typedef struct {
    int32_t device;             /* CUDA device ordinal */
    int32_t ref_len;            /* L: length of the reference genome */
    int32_t n_samples;          /* number of count matrices kept on the device (1; plate mode: many) */
    int32_t min_quality;        /* AmpliPy.py:27  */
    int32_t sliding_window;     /* AmpliPy.py:29  */
    int32_t min_length;         /* AmpliPy.py:26  */
    int32_t include_no_primer;  /* -e */
    int64_t ins_slots;          /* insertion hash table capacity (power of two; 0 = default) */
    int64_t ins_arena_bytes;    /* insertion string arena (0 = default) */
} amp_config;

typedef struct {
    int64_t first;              /* global index of the first read to process */
    int64_t n_reads;            /* reads to process: [first, first + n_reads) */
    const int32_t* pos; const uint16_t* flag; const int32_t* tlen;
    const uint32_t* cig_off; const uint32_t* cigar;
    const uint32_t* seq_off; const uint8_t* seq;
    const uint32_t* qual_off; const uint8_t* qual;
} amp_batch;

typedef struct {
    int32_t* pos;               /* [N] new reference_start (AmpliPy.py:514) */
    uint16_t* ncig;             /* [N] number of ops in the rewritten CIGAR */
    uint8_t* flags;             /* [N] AMP_FLAG_* */
    uint32_t* cigar;            /* [sumC + 3N] rows at cig_off[i] + 3*i */
} amp_trim_out;

typedef struct {
    int32_t min_depth_consensus; double min_freq_consensus;   /* AmpliPy.py:22,24 */
    int32_t min_depth_variants;  double min_freq_variants;    /* AmpliPy.py:23,25 */
} amp_call_params;

/* per-(sample, position) outputs of amp_call, host arrays of n_samples*L entries (x6 where noted) */
typedef struct {
    int32_t* depth;             /* total depth incl. insertion alleles (AmpliPy.py:767) */
    int32_t* top_id;            /* top allele: 0..5 = A C G T N '-', 6+k = insertion allele k of amp_ins_export order, -1 none */
    int32_t* top_count;
    uint8_t* pos_flags;         /* bit0 consensus passes (928); bit1 variant record emitted (940); bit2 GT includes ref (948) */
    int32_t* ref_count;         /* REF_DP (937) */
    double*  fixed_freq;        /* [.. x6] count/total as IEEE float64 */
    int32_t* fixed_rank;        /* [.. x6] index in the reference's sorted allele list (771), -1 if count 0 */
    uint8_t* alt_mask;          /* bit ch set: fixed symbol ch is an ALT allele (938) */
} amp_call_out;

const char* amp_last_error(void);
int amp_abi_version(void);

/* context: device tables + count matrices + insertion-allele table.  Primer tables are the two lists
 * returned by find_overlapping_primers (AmpliPy.py:174-209) with None encoded as -1; pass NULL for
 * pileup-only use (variants / consensus subcommands). */
int amp_create(const amp_config* cfg, const int32_t* min_primer_start, const int32_t* max_primer_end,
               int32_t max_primer_len, amp_ctx** out);
int amp_destroy(amp_ctx* ctx);
int amp_reset(amp_ctx* ctx);                          /* zero counts + insertion table + error word */
int amp_reset_async(amp_ctx* ctx, void* stream);      /* same, enqueued on `stream` without synchronising */
int amp_error_flags(amp_ctx* ctx, uint32_t* flags);   /* AMP_DEVERR_* accumulated since amp_reset */
int amp_lpad(amp_ctx* ctx);                           /* row stride of the count matrices (L rounded up to 32) */
int amp_sm_count(amp_ctx* ctx);

/* Replaces the per-read loop AmpliPy.py:896-915 for reads [first, first+n): trim_read + write gate,
 * and/or update_base_counts into count matrix `sample`.  Device-pointer variant: inputs already
 * resident in HBM; runs asynchronously on `stream`.  out may be NULL without AMP_MODE_TRIM.
 * sum_cigar_ops / sum_qual_bytes = totals over the processed range (known to the host that built the
 * batch); they size the long-CIGAR scratch and pick the shared-memory tile shape. */
int amp_process_device(amp_ctx* ctx, const amp_batch* dev_batch, int64_t sum_cigar_ops, int64_t sum_qual_bytes, int mode,
                       int sample, const amp_trim_out* dev_out, void* stream);
/* Host-buffer variant (the call a reference-side binding makes): chunks the batch, overlaps H2D copy,
 * kernel and D2H of the trim outputs on internal streams; returns when everything has landed. */
int amp_process_host(amp_ctx* ctx, const amp_batch* host_batch, int mode, int sample, const amp_trim_out* host_out);
int amp_last_launches(amp_ctx* ctx);                  /* kernels launched by the last amp_process_* / amp_call */

/* count matrices: device pointer [n_samples][6][lpad] int32 (channel order A C G T N '-'); copy to host */
int amp_counts_device(amp_ctx* ctx, int32_t** dev_counts);
int amp_bind_counts(amp_ctx* ctx, int32_t* dev_counts);          /* use a caller-owned device buffer (e.g. a torch tensor for NCCL) */
int amp_counts_host(amp_ctx* ctx, int sample, int32_t* host_counts /* [6][L] */);
int amp_counts_upload(amp_ctx* ctx, int sample, const int32_t* host_counts /* [6][L] */);   /* replace a sample's matrix */

/* insertion alleles (the non-fixed keys of symbol_counts_at_ref_pos, AmpliPy.py:745-748) */
int amp_ins_count(amp_ctx* ctx, int64_t* n_alleles, int64_t* n_chars);
int amp_ins_export(amp_ctx* ctx, int32_t* sample, int32_t* pos, int32_t* count, int64_t* str_off /* [n+1] */, char* chars);
/* add alleles produced elsewhere (another rank's amp_ins_export) into this context's table */
int amp_ins_merge(amp_ctx* ctx, int64_t n, const int32_t* sample, const int32_t* pos, const int32_t* count,
                  const int64_t* str_off, const char* chars);

/* Replaces alleles_from_counts + the calling loop (AmpliPy.py:756-771, 921-951) for every sample.
 * ref_seq: L raw FASTA characters.  Per-insertion-allele outputs are indexed like amp_ins_export.
 * The outputs are copied back as one queue of asynchronous copies followed by a single wait: destinations from
 * amp_host_alloc (page-locked) receive them at full PCIe speed, pageable ones work but are staged by the driver. */
int amp_call(amp_ctx* ctx, const char* ref_seq, const amp_call_params* p, const amp_call_out* host_out,
             double* ins_freq, int32_t* ins_rank, uint8_t* ins_alt);
/* the same kernels without the device->host copies: reference characters are uploaded once, results stay
 * in context-owned HBM buffers; asynchronous on `stream` */
int amp_set_reference(amp_ctx* ctx, const char* ref_seq);
int amp_call_device(amp_ctx* ctx, const amp_call_params* p, void* stream);

/* ---- iVar-format outputs (the reference has none; DESIGN.md 3.7).  amp_qstats_enable allocates and zeroes, per (sample, channel,
 * position), rev = the count matrix's increments from reverse-strand reads (flag & 0x10) and qsum = the phred qualities of the
 * counted A C G T N bases ('-' carries none), plus the same two sums per insertion allele (an event's quality = that of the first
 * inserted base past the gates 718 / 722).  amp_process_* with AMP_MODE_PILEUP | AMP_MODE_QSTATS then runs a second pass over the
 * same reads after the fused kernel; amp_reset / amp_reset_async zero the sums.  Across ranks the sums travel through the
 * *_qstats entry points of the deep-sample mode below; amp_allreduce_counts and amp_ins_pack_device, which would leave them
 * behind, return AMP_ERR_STATE on a context with them enabled.
 * amp_qstats_host: host arrays rev [6][L], qsum [6][L] of one sample, and ins_rev / ins_qsum / ins_head [n_alleles] in
 * amp_ins_export order (ins_head[k] = 1: an event of allele k is the key of AmpliPy.py:735-736); any pointer may be NULL.
 * amp_call_ivar (after amp_call): per allele mean quality mq = floor(qsum / count) ('-': the position's mean base quality) and,
 * for the alleles that get a TSV row (count > 0, symbol != the FASTA character, freq >= min_freq, depth >= min_depth; NaN
 * otherwise), PVAL = the left tail of Fisher's exact test on [[e, D - e], [a, D - a]], e = floor(D * 10^(-mq/10)); and per
 * (sample, position) an IUPAC code (0 = the reference's own consensus symbol) from the shortest prefix of the sorted allele
 * list whose frequencies reach iupac_threshold.  Per-allele outputs are indexed like amp_ins_export. */
typedef struct {
    int32_t min_depth; double min_freq;   /* TSV rows, and the consensus gate of AmpliPy.py:928 for the IUPAC code */
    double iupac_threshold;               /* [0, 1]; 0 = the reference's consensus */
} amp_ivar_params;
int amp_qstats_enable(amp_ctx* ctx);
int amp_qstats_host(amp_ctx* ctx, int sample, int32_t* rev, int64_t* qsum, int32_t* ins_rev, int64_t* ins_qsum, uint8_t* ins_head);
int amp_call_ivar(amp_ctx* ctx, const amp_ivar_params* p, uint8_t* iupac /* [S*L] */, int32_t* fixed_mq /* [S*L*6] */,
                  double* fixed_pval /* [S*L*6] */, int32_t* ins_mq, double* ins_pval);
/* the same kernel on the outputs amp_call_device left in HBM; results stay in context-owned buffers; asynchronous on `stream` */
int amp_call_ivar_device(amp_ctx* ctx, const amp_ivar_params* p, void* stream);

/* ---- anchored deletion alleles of the iVar TSV (DESIGN.md 3.7, --ivar_deletions).  An allele is (sample, anchor, len): a D op of
 * len bases directly after an M / = / X op of a read the pileup counted, in the CIGAR row it walked, whose last base (the anchor, at
 * reference position anchor = the D's start - 1) has quality >= min_quality.  Each carries count, rev (events from reads with flag &
 * 0x10) and qsum (the anchor qualities).  N ops and a D after S / I / P are not alleles; the '-' channel is unchanged.
 *   amp_dels_enable        allocate and zero an open-addressing table of `slots` slots (a power of two, rounded up; 0 = 2^20).
 *                          AMP_ERR_STATE without amp_qstats_enable: the strand / quality pass (AMP_MODE_QSTATS) fills it.  A
 *                          second call changes nothing.  A full table raises AMP_DEVERR_DELS_FULL.  amp_reset / amp_reset_async
 *                          clear it.
 *   amp_dels_count         the number of alleles
 *   amp_dels_export        the alleles sorted by (sample, anchor, len); any pointer may be NULL
 *   amp_dels_merge         host alleles added to the table (sums added to an existing allele's); AMP_ERR_ARG when one is out of range
 *   amp_call_ivar_dels     after amp_call: per allele in export order, mq = floor(qsum / count) and, when it gets a TSV row
 *                          (D > 0, D >= min_depth, count / D >= min_freq, D = depth at the anchor), PVAL as amp_call_ivar computes
 *                          it; NaN otherwise.  p->iupac_threshold is not used.
 * Every entry point returns AMP_ERR_STATE on a context without the table.  The deep-sample exchange of the table:
 *   amp_dels_slot_bytes    8 + 32 * cap_entries
 *   amp_dels_pack_device   { u64 n_alleles, {u64 key = (sample * lpad + anchor) << 32 | len, u64 count, u64 rev, u64 qsum}[cap_entries] };
 *                          a table of more than cap_entries alleles raises AMP_DEVERR_DELS_FULL and packs as empty
 *   amp_dels_merge_packed  the other ranks' alleles added to this rank's table (amp_nccl_allgather moves the slots) */
int amp_dels_enable(amp_ctx* ctx, int64_t slots);
int amp_dels_count(amp_ctx* ctx, int64_t* n_alleles);
int amp_dels_export(amp_ctx* ctx, int32_t* sample, int32_t* anchor, int32_t* len, int32_t* count, int32_t* rev, int64_t* qsum);
int amp_dels_merge(amp_ctx* ctx, int64_t n, const int32_t* sample, const int32_t* anchor, const int32_t* len, const int32_t* count,
                   const int32_t* rev, const int64_t* qsum);
int amp_call_ivar_dels(amp_ctx* ctx, const amp_ivar_params* p, int32_t* mq, double* pval);
int64_t amp_dels_slot_bytes(int64_t cap_entries);
int amp_dels_pack_device(amp_ctx* ctx, void* dev_slot, int64_t cap_entries, void* stream);
int amp_dels_merge_packed(amp_ctx* ctx, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries, void* stream);

/* ---- deep-sample mode: one sample's reads sharded over ranks (SURVEY.md 8e; the reference has no counterpart, its loop
 * AmpliPy.py:896-915 is sequential).  After every rank has processed its read range:
 *   amp_allreduce_counts  one ncclAllReduce(sum, int32) of the [n_samples][6][lpad] matrices, in place
 *   amp_ins_pack_device   this rank's insertion table -> one fixed-size slot in device memory
 *                         { u64 n_alleles, u64 arena_words, {u64 arena offset, u64 count}[cap_entries], arena[cap_arena_bytes] }
 *   (all-gather of the slots: amp_nccl_allgather, or any collective the host prefers)
 *   amp_ins_merge_packed  everybody else's alleles added to this rank's table by one kernel
 * Everything is asynchronous on `stream`; nothing allocates.  A table that does not fit its slot raises
 * AMP_DEVERR_TABLE_FULL / AMP_DEVERR_ARENA_FULL (amp_error_flags) and packs as empty.
 * NCCL is resolved with dlopen at the first call (libnccl.so.2 as already mapped by the process, else the system's;
 * AMP_NCCL_LIB overrides); `comm` is an ncclComm_t, from amp_nccl_comm_init or the caller's own ncclCommInitRank. */
int amp_nccl_unique_id(uint8_t* id128 /* [128] */);
int amp_nccl_comm_init(int device, int n_ranks, int rank, const uint8_t* id128, void** comm);
int amp_nccl_comm_destroy(void* comm);
int amp_nccl_allgather(void* comm, const void* dev_send, void* dev_recv, int64_t bytes_per_rank, void* stream);
int amp_allreduce_counts(amp_ctx* ctx, void* comm, void* stream);
int64_t amp_ins_slot_bytes(int64_t cap_entries, int64_t cap_arena_bytes);
int amp_ins_pack_device(amp_ctx* ctx, void* dev_slot, int64_t cap_entries, int64_t cap_arena_bytes, void* stream);
int amp_ins_merge_packed(amp_ctx* ctx, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries,
                         int64_t cap_arena_bytes, void* stream);
/* The same exchange for a context with the strand / quality sums (amp_qstats_enable); each returns AMP_ERR_STATE on a context
 * without them (and amp_allreduce_qstats does so before it calls NCCL).  Afterwards every rank holds what one context over all the
 * reads would hold: counts, insertion alleles, rev / qsum and each allele's ins_rev / ins_qsum / ins_head.
 *   amp_allreduce_qstats         three ncclAllReduce(sum), in place: counts and rev (int32), qsum (uint64)
 *   amp_ins_slot_bytes_qstats    16 + 32 * cap_entries + cap_arena_bytes rounded up to 8
 *   amp_ins_pack_qstats_device   { u64 n_alleles, u64 arena_words,
 *                                  {u64 arena offset, u64 count, u64 ins_qsum, u64 ins_rev | ins_head << 32}[cap_entries],
 *                                  arena[cap_arena_bytes] }; the same overflow contract as amp_ins_pack_device
 *   amp_ins_merge_packed_qstats  the other ranks' alleles with their sums; an allele the table cannot take gets no sums (the
 *                                TABLE_FULL / ARENA_FULL bit reports the loss) */
int amp_allreduce_qstats(amp_ctx* ctx, void* comm, void* stream);
int64_t amp_ins_slot_bytes_qstats(int64_t cap_entries, int64_t cap_arena_bytes);
int amp_ins_pack_qstats_device(amp_ctx* ctx, void* dev_slot, int64_t cap_entries, int64_t cap_arena_bytes, void* stream);
int amp_ins_merge_packed_qstats(amp_ctx* ctx, const void* dev_slots, int n_ranks, int my_rank, int64_t cap_entries,
                                int64_t cap_arena_bytes, void* stream);

/* pre-size what amp_process_device would otherwise grow on demand (it synchronises `stream` when it has to allocate) */
int amp_reserve(amp_ctx* ctx, int64_t max_reads, int64_t max_cigar_ops);
/* device-to-device copy of the count matrices into a caller-owned buffer of the same shape */
int amp_counts_copy_device(amp_ctx* ctx, int32_t* dev_dst, void* stream);

/* ---- BAM on the device (SURVEY.md 8f-1; replaces pysam's record iteration, AmpliPy.py:296-360 + 896, in front of the path).
 * The compressed file crosses PCIe as it is (about a fifth of the decoded arrays) and is decoded in HBM: one warp inflates one
 * BGZF block (RFC 1951), one thread per block walks its BAM record chain, one warp per block scatters the records into the
 * struct-of-arrays batch the kernels read.  Requires what htslib guarantees for the files it writes: no record straddles a BGZF
 * block boundary; otherwise AMP_ERR_DATA is returned and the caller uses its host decoder.  CRC32 of the blocks is not checked
 * on the device (ISIZE is).
 *   bgzf, n_bytes      the file's bytes (page-locked memory makes the copy asynchronous)
 *   block_off[n_blocks], block_isize[n_blocks]   start of every BGZF block in `bgzf` and its ISIZE (a host-side header scan)
 *   body_off           offset of the first alignment record in the inflated stream (= size of the BAM header)
 * amp_process_decoded runs the fused kernel on the decoded batch and copies the trim outputs (rows as in amp_trim_out,
 * sized from amp_bam_info) to host_out; host_out may be NULL.  amp_decoded_copy_host hands the decoded arrays back. */
typedef struct { int64_t n_reads, sum_cigar_ops, sum_seq_bytes, sum_qual_bytes, raw_bytes; } amp_bam_info;
typedef struct {
    int32_t* pos; uint16_t* flag; int32_t* tlen; uint32_t* cig_off; uint32_t* cigar; uint32_t* seq_off; uint8_t* seq;
    uint32_t* qual_off; uint8_t* qual;
} amp_batch_out;
int amp_bam_decode_host(amp_ctx* ctx, const uint8_t* bgzf, int64_t n_bytes, const int64_t* block_off, const uint32_t* block_isize,
                        int64_t n_blocks, int64_t body_off, amp_bam_info* info);
int amp_process_decoded(amp_ctx* ctx, int mode, int sample, const amp_trim_out* host_out);
int amp_decoded_copy_host(amp_ctx* ctx, const amp_batch_out* host_arrays, uint64_t* rec_off);

/* ---- BGZF deflate on the device (SURVEY.md 8f-2; replaces the zlib deflate behind out_aln.write, AmpliPy.py:911).
 * host data -> BGZF blocks: block k = in[bstart[k], bstart[k + 1]) (bstart has n_blocks + 1 entries, bstart[0] = 0, the last one =
 * n_bytes, every block at most 0xff00 bytes -- the caller cuts at record boundaries as htslib does), followed by the EOF block.
 * One warp per block: LZ77 (4-byte hash + run candidate), a Huffman code built for every 8 k tokens (or the fixed code where that is
 * shorter), CRC-32 and ISIZE in the footer; a block that does not shrink is stored.  Any inflater reads the result; it is a little
 * smaller than zlib level 1 writes.
 * out must hold n_bytes + 31 * n_blocks + 28 bytes.  Returns the number of bytes written, or a negative AMP_ERR_* code. */
int64_t amp_bgzf_deflate_host(amp_ctx* ctx, const uint8_t* in, int64_t n_bytes, const int64_t* bstart, int64_t n_blocks, uint8_t* out,
                              int64_t out_cap);

/* The trimmed BAM file of the decoded batch, built on the device (replaces the cigartuples / reference_start assignments and
 * out_aln.write of AmpliPy.py:463-658, 910-911 for BAM input): after amp_bam_decode_host + amp_process_decoded(AMP_MODE_TRIM) the
 * inflated input and the trim outputs are both in HBM; the records of the reads that pass the write gate are rebuilt there (new
 * block_size / pos / bin / n_cigar / CIGAR, the rest byte for byte), cut into BGZF blocks at record boundaries, compressed
 * (amp_bgzf_deflate_host's kernels) and copied to the host once.  header = the BAM header the file starts with (magic, l_text,
 * text, references).  out must hold header_bytes + the inflated input + 31 bytes per 64 KB + 28.  Returns the size of the file
 * or a negative AMP_ERR_* code; *n_records = the number of records written. */
int64_t amp_decoded_write_bam(amp_ctx* ctx, const uint8_t* header, int64_t header_bytes, uint8_t* out, int64_t out_cap, int64_t* n_records);

/* ---- heterogeneous plates (SURVEY.md 8f-4): a primer scheme and / or a reference of its own for one sample of the context.
 * amp_set_scheme builds the two per-position tables of find_overlapping_primers (AmpliPy.py:174-209) on the device from the
 * sorted primer list (start, end) and the offset; ref_len <= the context's ref_len.  amp_process_* of that sample then trims
 * against these tables, amp_call calls it against its own reference; one calling launch still covers the whole plate. */
int amp_set_scheme(amp_ctx* ctx, int sample, int32_t ref_len, const int32_t* primer_start, const int32_t* primer_end,
                   int32_t n_primers, int32_t offset);
int amp_get_scheme(amp_ctx* ctx, int sample, int32_t* min_primer_start, int32_t* max_primer_end, int32_t* max_primer_len);
int amp_set_sample_reference(amp_ctx* ctx, int sample, const char* ref_seq, int32_t len);

/* ---- multi-contig references (DESIGN.md 3.8): contig k of the FASTA is sample k of the context, with its own scheme
 * (amp_set_scheme with ref_len = the contig's length; n_primers may be 0) and reference (amp_set_sample_reference).
 * A plan call finds every read's contig -- the BAM record's refID through ref_to_sample (-1: no contig, -2: a header sequence
 * that is not in the FASTA) for the decoded batch, or a per-read sample id in [-1, n_samples) for a device batch -- and
 * returns per-contig totals.  A read without a contig must carry flag 4; it is trimmed as the fused kernels trim a read that
 * AmpliPy.py:902 skips and is not piled up.  The context holds at most AMP_MAX_CONTIGS = 1024 samples for this
 * (AMP_ERR_ARG beyond).  amp_process_contigs then runs the fused kernel (and, with AMP_MODE_QSTATS, the strand / quality pass)
 * once per contig with reads, over that contig's reads in input order: directly on the batch when it is grouped (every
 * contig's reads contiguous, as in any coordinate-sorted BAM), else on a copy reordered by a stable counting sort, whose trim
 * outputs are written back to input order.  Trim outputs: the decoded batch keeps them in the context (dev_out = NULL;
 * amp_decoded_write_bam reads them), a device batch writes them to dev_out; host_out (may be NULL) receives a copy.
 * amp_process_contigs returns AMP_ERR_DATA when the plan has error bits, and runs on the batch planned last. */
#define AMP_CONTIG_E_NOFLAG4 1     /* a read without a contig is not flagged unmapped (flag 4) */
#define AMP_CONTIG_E_UNKNOWN 2     /* a read on a header sequence that is not in the FASTA (ref_reads says which) */
#define AMP_CONTIG_E_BADID 4       /* refID outside the header, or a sample id outside [-1, n_samples) */
typedef struct {
    int64_t n_reads;            /* out: reads in the batch */
    int64_t n_no_contig;        /* out: reads without a contig */
    int32_t grouped;            /* out: 1 = every contig's reads are contiguous */
    uint32_t errors;            /* out: AMP_CONTIG_E_* */
    int64_t* contig_reads;      /* [n_samples] out (caller-owned; any of these may be NULL): reads of contig k */
    int64_t* contig_first;      /*   index of its first read */
    int64_t* contig_cigar_ops;  /*   CIGAR ops of its reads */
    int64_t* contig_qual_bytes; /*   quality bytes of its reads */
    int64_t* ref_reads;         /* [n_refs] out, decoded plan only: reads on header sequence r when ref_to_sample[r] = -2 */
} amp_contig_plan;
int amp_contig_plan_decoded(amp_ctx* ctx, const int32_t* ref_to_sample, int32_t n_refs, amp_contig_plan* plan);
int amp_contig_plan_device(amp_ctx* ctx, const amp_batch* dev_batch /* first = 0 */, const int32_t* dev_sample_of_read,
                           amp_contig_plan* plan);
int amp_process_contigs(amp_ctx* ctx, int mode, const amp_trim_out* dev_out, const amp_trim_out* host_out);

/* ---- codon annotation of the iVar TSV (DESIGN.md 3.9): the CDS features of a GFF3 file, per sample.
 * amp_set_features gives sample `sample` its features: feature f has strand[f] (+1 / -1), phase[f] (0..2: bases skipped before
 * its first codon), and the segments [seg_off[f], seg_off[f + 1]) of seg_start / seg_end (0-based, half-open, in any order: they
 * are spliced 5' to 3').  Checked against the sample's reference length (amp_set_reference / amp_set_sample_reference first,
 * else AMP_ERR_STATE); bad input is AMP_ERR_ARG.  n_features = 0 clears the sample.
 * amp_annotate builds, on the device, the occurrences of every (sample, position): the (feature, codon) pairs it belongs to,
 * in feature order, then in spliced order, as CSR over S*L positions, with each one's reference codon and amino acid and the
 * codon and amino acid of every substitution A C G T N at the position (standard code, table 1; '*' stop, 'X' any codon with
 * a character other than ACGT).  *n_entries = the number of occurrences.  AMP_ERR_STATE without features.
 * amp_annot_host copies the result: off[S*L + 1] (occurrences of position gp: [off[gp], off[gp + 1])), and per occurrence the
 * feature's index in its sample, the 1-based codon index, the position's offset in the codon, 18 codon characters (REF, then
 * ALT for A C G T N) and 6 amino acids (the same order); any pointer may be NULL.  AMP_ERR_STATE unless amp_annotate ran after
 * the last change of features or reference. */
int amp_set_features(amp_ctx* ctx, int sample, int32_t n_features, const int32_t* strand, const int32_t* phase, const int32_t* seg_off,
                     const int32_t* seg_start, const int32_t* seg_end);
int amp_annotate(amp_ctx* ctx, int64_t* n_entries);
int amp_annot_host(amp_ctx* ctx, uint32_t* off, int32_t* feat, int32_t* pos_aa, uint8_t* codon_off, char* codons, char* aas);

/* pinned host memory helpers for callers that want full-speed amp_process_host */
int amp_host_alloc(void** p, int64_t bytes);
int amp_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif
