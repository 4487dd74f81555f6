// amp_emu_contig.cpp -- TEST INFRASTRUCTURE: the grouping of a batch by contig (amp_contig.cuh), the kernels' own source run on the
// CPU with every CUDA thread a fiber of the emulator's runtime (amp_emu.cpp).  Not part of the product.
#include "amp_emu.cpp"
#include "../../amplipy_b200/csrc/amp_contig.cuh"

namespace {
template <class F>
void run_grid(long long blocks, int nthreads, F f) {       // the CTAs one after another, f(block) on every fiber of each
    struct Arg { F* f; int block; } a{&f, 0};
    for (long long b = 0; b < blocks; ++b) {
        a.block = (int)b;
        run_cta((int)b, nthreads, [](void* p) { Arg* x = (Arg*)p; (*x->f)(x->block); }, &a);
    }
}
}  // namespace

extern "C" {

// amp_contig_plan_kernel over every tile; table: ct_table_words(S, n_refs) u64, zeroed here
void emu_contig_plan(long long n, const uint8_t* raw, const unsigned long long* rec_off, const int* ref_to_sample, int n_refs,
                     const int* sample_in, const uint16_t* flag, const uint32_t* cig_off, const uint32_t* qual_off, int S, int* sid,
                     uint32_t* tile_hist, unsigned long long* table, int nthreads) {
    amp::ContigPlanParams P{};
    P.n = n; P.raw = raw; P.rec_off = rec_off; P.ref_to_sample = ref_to_sample; P.n_refs = n_refs; P.sample_in = sample_in;
    P.flag = flag; P.cig_off = cig_off; P.qual_off = qual_off; P.S = S; P.sid = sid; P.tile_hist = tile_hist; P.table = table;
    memset(table, 0, amp::ct_table_words(S, n_refs) * 8);
    static amp::ContigPlanSmem sm;
    run_grid((n + AMP_CT_TILE - 1) / AMP_CT_TILE, nthreads, [&](int b) { amp::contig_plan_cta(P, sm, b); });
}

// the launches of contig_permute (amp_abi.cu): contig-major scan of the tile histograms, rank, tile sums, their scans, gather
void emu_contig_permute(long long n, int S, const int* sid, const uint32_t* tile_hist, long long n_in, const int32_t* pos,
                        const uint16_t* flag, const int32_t* tlen, const uint32_t* cig_off, const uint32_t* cigar, const uint32_t* seq_off,
                        const uint8_t* seq, const uint32_t* qual_off, const uint8_t* qual, uint32_t* perm, int32_t* o_pos, uint16_t* o_flag,
                        int32_t* o_tlen, uint32_t* o_cig_off, uint32_t* o_cigar, uint32_t* o_seq_off, uint8_t* o_seq, uint32_t* o_qual_off,
                        uint8_t* o_qual, int nthreads) {
    const long long n_tiles = (n + AMP_CT_TILE - 1) / AMP_CT_TILE, pt = (n_in + AMP_CT_TILE - 1) / AMP_CT_TILE;
    static unsigned long long part[AMP_CT_THREADS];
    std::vector<uint32_t> hist_off((size_t)S * n_tiles + 1), tsum((size_t)pt * 3 + 3), tbase(3 * ((size_t)pt + 1));
    amp::ContigScanParams H{tile_hist, (long long)S * n_tiles, n_tiles, (long long)S, 1, hist_off.data()};
    run_grid(1, nthreads, [&](int) { amp::contig_scan_cta(H, part); });
    amp::ContigRankParams R{n, S, n_tiles, sid, hist_off.data(), perm};
    static amp::ContigRankSmem rsm;
    run_grid(n_tiles, nthreads, [&](int b) { amp::contig_rank_cta(R, rsm, b); });
    amp::ContigGatherParams G{};
    G.n = n_in; G.n_tiles = pt; G.perm = perm;
    G.src = amp::BatchPtrs{0, n, pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual};
    G.pos = o_pos; G.flag = o_flag; G.tlen = o_tlen; G.cig_off = o_cig_off; G.cigar = o_cigar; G.seq_off = o_seq_off; G.seq = o_seq;
    G.qual_off = o_qual_off; G.qual = o_qual; G.tsum = tsum.data(); G.tbase = tbase.data();
    if (n_in == 0) { o_cig_off[0] = o_seq_off[0] = o_qual_off[0] = 0; return; }
    run_grid(pt, nthreads, [&](int b) { amp::contig_tilesum_cta(G, part, b); });
    for (int ch = 0; ch < 3; ++ch) {
        amp::ContigScanParams Q{tsum.data() + ch, pt, pt, 3, 0, tbase.data() + (size_t)ch * (pt + 1)};
        run_grid(1, nthreads, [&](int) { amp::contig_scan_cta(Q, part); });
    }
    run_grid(pt, nthreads, [&](int b) { amp::contig_gather_cta(G, part, b); });
}

// amp_contig_unpermute_kernel with `blocks` CTAs of nthreads
void emu_contig_unpermute(long long n_in, const uint32_t* perm, const uint32_t* pcig_off, const int32_t* po_pos, const uint16_t* po_ncig,
                          const uint8_t* po_flags, const uint32_t* po_cigar, const uint32_t* cig_off, int32_t* o_pos, uint16_t* o_ncig,
                          uint8_t* o_flags, uint32_t* o_cigar, int blocks, int nthreads) {
    amp::ContigUnpermuteParams U{n_in, perm, pcig_off, amp::TrimOut{const_cast<int32_t*>(po_pos), const_cast<uint16_t*>(po_ncig),
                                 const_cast<uint8_t*>(po_flags), const_cast<uint32_t*>(po_cigar)}, cig_off, amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar}};
    const long long nw = (long long)blocks * nthreads / 32;
    run_grid(blocks, nthreads, [&](int b) { amp::contig_unpermute_warp(U, ((long long)b * nthreads + amp::c_tid()) >> 5, nw); });
}

void emu_contig_skip(long long n, const int* sid, const int32_t* pos, const uint32_t* cig_off, const uint32_t* cigar, int32_t* o_pos,
                     uint16_t* o_ncig, uint8_t* o_flags, uint32_t* o_cigar) {
    amp::ContigSkipParams K{};
    K.n = n; K.sid = sid; K.b.pos = pos; K.b.cig_off = cig_off; K.b.cigar = cigar; K.o = amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar};
    for (long long i = 0; i < n; ++i) amp::contig_skip_read(K, i);
}

}  // extern "C"
