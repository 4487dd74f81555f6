// amp_emu.cpp -- TEST INFRASTRUCTURE: runs the CUDA kernels' own source (amplipy_b200/csrc/*.cuh) on the
// CPU, one CTA at a time with barrier-separated phases executed as loops over the CTA's threads.
// It lets the build container (no GPU) check the device logic against the oracle before a GPU run.
// It is not part of the product and is never loaded by amplipy_b200/.
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <ucontext.h>

#include <cstdio>

#include "../../amplipy_b200/csrc/amp_warp.cuh"
#include "../../amplipy_b200/csrc/amp_bgzf.cuh"
#include "../../amplipy_b200/csrc/amp_ont.cuh"
#include "../../amplipy_b200/csrc/amp_deflate.cuh"

// ---------------------------------------------------------------------------------------------------------------------
// Fiber runtime for the warp-autonomous kernel: every CUDA thread of one CTA is a ucontext fiber; warp collectives
// (shuffle, ballot, reduce, __syncwarp) and the block barrier are rendezvous points handled by a round-robin scheduler.
// Deterministic and single-threaded, so shared-memory "atomics" can stay plain read-modify-writes.
// ---------------------------------------------------------------------------------------------------------------------
namespace {
enum { FB_READY = 0, FB_WAIT_WARP = 1, FB_WAIT_CTA = 2, FB_DONE = 3 };
struct Fiber { ucontext_t ctx; int state; };
struct FiberRt {
    std::vector<Fiber> f;
    std::vector<char> stacks;
    ucontext_t main_ctx;
    int cur = 0, nthreads = 0, block = 0;
    int xch[1024];
    void (*body)(void*) = nullptr;
    void* arg = nullptr;
} g_rt;
const size_t kStack = 256 * 1024;

void fiber_entry() {
    g_rt.body(g_rt.arg);
    g_rt.f[g_rt.cur].state = FB_DONE;
    swapcontext(&g_rt.f[g_rt.cur].ctx, &g_rt.main_ctx);
}
void fiber_wait(int kind) {
    g_rt.f[g_rt.cur].state = kind;
    swapcontext(&g_rt.f[g_rt.cur].ctx, &g_rt.main_ctx);
}
void run_cta(int block, int nthreads, void (*body)(void*), void* arg) {
    g_rt.block = block; g_rt.nthreads = nthreads; g_rt.body = body; g_rt.arg = arg;
    g_rt.f.assign(nthreads, Fiber());
    if (g_rt.stacks.size() < kStack * nthreads) g_rt.stacks.resize(kStack * nthreads);
    for (int t = 0; t < nthreads; ++t) {
        getcontext(&g_rt.f[t].ctx);
        g_rt.f[t].ctx.uc_stack.ss_sp = g_rt.stacks.data() + kStack * t;
        g_rt.f[t].ctx.uc_stack.ss_size = kStack;
        g_rt.f[t].ctx.uc_link = &g_rt.main_ctx;
        g_rt.f[t].state = FB_READY;
        makecontext(&g_rt.f[t].ctx, fiber_entry, 0);
    }
    for (;;) {
        bool progress = false, all_done = true;
        for (int t = 0; t < nthreads; ++t) {
            if (g_rt.f[t].state == FB_READY) {
                g_rt.cur = t;
                swapcontext(&g_rt.main_ctx, &g_rt.f[t].ctx);
                progress = true;
            }
            if (g_rt.f[t].state != FB_DONE) all_done = false;
        }
        if (all_done) break;
        // release warps whose live lanes all wait at a warp rendezvous
        for (int w = 0; w * 32 < nthreads; ++w) {
            int waiting = 0, live = 0;
            for (int t = w * 32; t < std::min(nthreads, w * 32 + 32); ++t) {
                if (g_rt.f[t].state != FB_DONE) ++live;
                if (g_rt.f[t].state == FB_WAIT_WARP) ++waiting;
            }
            if (live && waiting == live) {
                for (int t = w * 32; t < std::min(nthreads, w * 32 + 32); ++t) if (g_rt.f[t].state == FB_WAIT_WARP) g_rt.f[t].state = FB_READY;
                progress = true;
            }
        }
        {
            int waiting = 0, live = 0;
            for (int t = 0; t < nthreads; ++t) {
                if (g_rt.f[t].state != FB_DONE) ++live;
                if (g_rt.f[t].state == FB_WAIT_CTA) ++waiting;
            }
            if (live && waiting == live) {
                for (int t = 0; t < nthreads; ++t) g_rt.f[t].state = FB_READY;
                progress = true;
            }
        }
        if (!progress) { fprintf(stderr, "amp_emu: deadlock in the fiber runtime (divergent collective?)\n"); abort(); }
    }
}
}  // namespace

namespace amp {
int c_tid() { return g_rt.cur; }
int c_nthreads() { return g_rt.nthreads; }
int c_block() { return g_rt.block; }
void w_sync() { fiber_wait(FB_WAIT_WARP); }
void c_sync() { fiber_wait(FB_WAIT_CTA); }
void c_yield() { fiber_wait(FB_READY); }             // spin-wait: let the other fibers run
int w_shfl(int v, int src) {
    g_rt.xch[g_rt.cur] = v;
    w_sync();
    const int r = g_rt.xch[(g_rt.cur & ~31) | (src & 31)];
    w_sync();
    return r;
}
unsigned w_ballot(bool p) {
    g_rt.xch[g_rt.cur] = p ? 1 : 0;
    w_sync();
    unsigned r = 0;
    for (int k = 0; k < 32; ++k) if ((g_rt.cur & ~31) + k < g_rt.nthreads && g_rt.xch[(g_rt.cur & ~31) + k]) r |= 1u << k;
    w_sync();
    return r;
}
int w_add(int v) {
    g_rt.xch[g_rt.cur] = v;
    w_sync();
    int r = 0;
    for (int k = 0; k < 32; ++k) if ((g_rt.cur & ~31) + k < g_rt.nthreads) r += g_rt.xch[(g_rt.cur & ~31) + k];
    w_sync();
    return r;
}
}  // namespace amp

struct EmuCtx {
    int L, Lpad, n_samples;
    amp::TrimParams tp;
    std::vector<int32_t> mn, mx;
    std::vector<int> counts;
    std::vector<amp::InsSlot> slots;
    std::vector<unsigned int> entries;
    std::vector<int> slot_entry;
    std::vector<unsigned char> arena;
    unsigned long long cursor[2];
    unsigned int err;
    amp::InsTable tab;
};

extern "C" {

void* emu_create(int L, int n_samples, const int32_t* mn, const int32_t* mx, int max_primer_len, int min_quality, int window,
                 int min_length, int include_no_primer, long long nslots, long long arena_bytes) {
    EmuCtx* c = new EmuCtx();
    c->L = L; c->Lpad = (L + 31) & ~31; c->n_samples = n_samples;
    if (mn) { c->mn.assign(mn, mn + L); c->mx.assign(mx, mx + L); }
    c->tp.L = L; c->tp.min_primer_start = mn ? c->mn.data() : nullptr; c->tp.max_primer_end = mn ? c->mx.data() : nullptr;
    c->tp.max_primer_len = max_primer_len; c->tp.min_quality = min_quality; c->tp.window = window;
    c->tp.min_length = min_length; c->tp.include_no_primer = include_no_primer;
    c->counts.assign((size_t)n_samples * AMP_NCH * c->Lpad, 0);
    c->slots.assign(nslots, amp::InsSlot{0, 0, 0});
    c->entries.assign(nslots, 0); c->slot_entry.assign(nslots, 0);
    c->arena.assign(arena_bytes, 0);
    c->cursor[0] = c->cursor[1] = 0; c->err = 0;
    c->tab.slots = c->slots.data(); c->tab.mask = (unsigned long long)nslots - 1; c->tab.entries = c->entries.data();
    c->tab.slot_entry = c->slot_entry.data(); c->tab.arena = c->arena.data(); c->tab.arena_words = arena_bytes / 8;
    c->tab.cursor = c->cursor; c->tab.err = &c->err;
    return c;
}
void emu_destroy(void* h) { delete (EmuCtx*)h; }
unsigned int emu_error_flags(void* h) { return ((EmuCtx*)h)->err; }
// as amp_reset_kernel: zero counts, the slots listed in entries[0, cursor[1]), both cursors and the error word; the arena
// keeps its bytes
void emu_reset(void* h) {
    EmuCtx* c = (EmuCtx*)h;
    std::fill(c->counts.begin(), c->counts.end(), 0);
    for (unsigned long long k = 0; k < c->cursor[1]; ++k) c->slots[c->entries[k]] = amp::InsSlot{0, 0, 0};
    c->cursor[0] = c->cursor[1] = 0; c->err = 0;
}

// grid / threads / reads_per_tile overrides (0 = what the product's launch code would choose)
int emu_process(void* h, long long first, long long n, const int32_t* pos, const uint16_t* flag, const int32_t* tlen,
                const uint32_t* cig_off, const uint32_t* cigar, const uint32_t* seq_off, const uint8_t* seq,
                const uint32_t* qual_off, const uint8_t* qual, int mode, int sample, int32_t* o_pos, uint16_t* o_ncig,
                uint8_t* o_flags, uint32_t* o_cigar, int grid_override, int threads, int rpt_override, int maxseg_override,
                int wt_override, int qbytes_override) {
    EmuCtx* c = (EmuCtx*)h;
    amp::KParams P{};
    P.b = amp::BatchPtrs{first, n, pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual};
    P.o = amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar};
    P.tp = c->tp; P.mode = mode;
    P.counts = c->counts.data() + (size_t)sample * AMP_NCH * c->Lpad; P.Lpad = c->Lpad; P.gpos_base = sample * c->Lpad;
    P.tab = c->tab; P.err = &c->err;
    const long long sum_cig = cig_off[first + n] - cig_off[first];
    std::vector<uint32_t> scratch(2 * (size_t)(sum_cig + 3 * n) + 8);
    P.scratch = scratch.data() - ((size_t)cig_off[first] + 3 * (size_t)first);
    P.scratch_half = sum_cig + 3 * n;
    amp::TileCfg t = amp::pick_tile_cfg(n, sum_cig, (long long)(qual_off[first + n] - qual_off[first]), mode);
    if (rpt_override) t.reads_per_tile = rpt_override;
    if (maxseg_override) t.maxseg = maxseg_override;
    if (wt_override) t.wt = wt_override;
    if (qbytes_override) { t.qbytes = qbytes_override; t.sbytes = qbytes_override / 2; }
    P.wt = t.wt; P.maxseg = t.maxseg; P.qbytes = t.qbytes; P.sbytes = t.sbytes; P.reads_per_tile = t.reads_per_tile;
    P.ntiles = (int)((n + t.reads_per_tile - 1) / t.reads_per_tile);
    int grid = grid_override ? grid_override : 296;
    if (grid > P.ntiles) grid = P.ntiles;
    if (grid < 1) grid = 1;
    P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
    grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
    std::vector<unsigned char> smem(amp::smem_bytes(P.wt, P.maxseg, P.qbytes, P.sbytes) + 64);
    unsigned char* sbase = smem.data();
    sbase += (16 - ((uintptr_t)sbase & 15)) & 15;
    P.direct = t.direct;
    for (int b = 0; b < grid; ++b) {
        if (P.direct) amp::cta_trim_pileup<true>(P, sbase, b, threads ? threads : 256);
        else amp::cta_trim_pileup<false>(P, sbase, b, threads ? threads : 256);
    }
    return 0;
}

// the warp-autonomous kernel (amp_warp.cuh): one CTA at a time, every thread a fiber
struct V7Launch { const amp::KParams* P; unsigned char* smem; int mode, gwarps, dwarps; };
static void v9_body(void* a) {
    V7Launch* v = (V7Launch*)a;
    if (v->mode == 3) amp::cta_trim_pileup_v9<true, true, 0>(*v->P, v->smem, v->gwarps, v->dwarps);
    else if (v->mode == 1) amp::cta_trim_pileup_v9<true, false, 0>(*v->P, v->smem, v->gwarps, v->dwarps);
    else amp::cta_trim_pileup_v9<false, true, 0>(*v->P, v->smem, v->gwarps, v->dwarps);
}
int emu_process_v7(void* h, long long first, long long n, const int32_t* pos, const uint16_t* flag, const int32_t* tlen,
                   const uint32_t* cig_off, const uint32_t* cigar, const uint32_t* seq_off, const uint8_t* seq,
                   const uint32_t* qual_off, const uint8_t* qual, int mode, int sample, int32_t* o_pos, uint16_t* o_ncig,
                   uint8_t* o_flags, uint32_t* o_cigar, int grid_override, int warps, int br_override, int wt_override) {
    EmuCtx* c = (EmuCtx*)h;
    if (n <= 0) return 0;
    amp::KParams P{};
    P.b = amp::BatchPtrs{first, n, pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual};
    P.o = amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar};
    P.tp = c->tp; P.mode = mode;
    P.counts = c->counts.data() + (size_t)sample * AMP_NCH * c->Lpad; P.Lpad = c->Lpad; P.gpos_base = sample * c->Lpad;
    P.tab = c->tab; P.err = &c->err;
    const long long sum_cig = cig_off[first + n] - cig_off[first];
    std::vector<uint32_t> scratch(2 * (size_t)(sum_cig + 3 * n) + 8);
    P.scratch = scratch.data() - ((size_t)cig_off[first] + 3 * (size_t)first);
    P.scratch_half = sum_cig + 3 * n;
    const amp::V7Cfg t = amp::pick_v7_cfg(n, (long long)(qual_off[first + n] - qual_off[first]), grid_override ? grid_override : 148);
    P.wt = wt_override ? wt_override : t.wt;
    P.reads_per_tile = br_override ? br_override : t.batch_reads;
    P.ntiles = (int)((n + P.reads_per_tile - 1) / P.reads_per_tile);
    int grid = std::max(1, std::min(grid_override ? grid_override : 148, P.ntiles));
    P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
    grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
    if (!warps) warps = AMP7_WARPS;
    const int gwarps = std::max(1, std::min(warps, AMP7_GWARPS));
    std::vector<unsigned char> smem(amp::smem_bytes_v9(P.wt, warps, gwarps) + 64);
    unsigned char* sbase = smem.data();
    sbase += (16 - ((uintptr_t)sbase & 15)) & 15;
    P.gcap = (long long)P.tiles_per_cta * P.reads_per_tile;
    std::vector<uint32_t> glist((size_t)grid * P.gcap + 1);
    P.glist = glist.data();
    const int dwarps = warps >= 3 ? 1 : 0;              // one dedicated list warp when there are warps to spare
    V7Launch v{&P, sbase, mode, gwarps, dwarps};
    for (int b = 0; b < grid; ++b) run_cta(b, warps * 32, v9_body, &v);
    return 0;
}

// the warp-per-read kernel for indel-rich batches (amp_ont.cuh)
struct OntLaunch { const amp::KParams* P; unsigned char* smem; int mode, gwarps; };
static void ont_body(void* a) {
    OntLaunch* v = (OntLaunch*)a;
    if (v->mode == 3) amp::cta_trim_pileup_ont<true, true, 0>(*v->P, v->smem, v->gwarps);
    else if (v->mode == 1) amp::cta_trim_pileup_ont<true, false, 0>(*v->P, v->smem, v->gwarps);
    else amp::cta_trim_pileup_ont<false, true, 0>(*v->P, v->smem, v->gwarps);
}
int emu_process_ont(void* h, long long first, long long n, const int32_t* pos, const uint16_t* flag, const int32_t* tlen,
                    const uint32_t* cig_off, const uint32_t* cigar, const uint32_t* seq_off, const uint8_t* seq,
                    const uint32_t* qual_off, const uint8_t* qual, int mode, int sample, int32_t* o_pos, uint16_t* o_ncig,
                    uint8_t* o_flags, uint32_t* o_cigar, int grid_override, int warps, int wt_override) {
    EmuCtx* c = (EmuCtx*)h;
    if (n <= 0) return 0;
    amp::KParams P{};
    P.b = amp::BatchPtrs{first, n, pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual};
    P.o = amp::TrimOut{o_pos, o_ncig, o_flags, o_cigar};
    P.tp = c->tp; P.mode = mode;
    P.counts = c->counts.data() + (size_t)sample * AMP_NCH * c->Lpad; P.Lpad = c->Lpad; P.gpos_base = sample * c->Lpad;
    P.tab = c->tab; P.err = &c->err;
    const long long sum_cig = cig_off[first + n] - cig_off[first];
    std::vector<uint32_t> scratch(2 * (size_t)(sum_cig + 3 * n) + 8);
    P.scratch = scratch.data() - ((size_t)cig_off[first] + 3 * (size_t)first);
    P.scratch_half = sum_cig + 3 * n;
    P.wt = wt_override ? wt_override : AMPO_WT;
    P.reads_per_tile = 1; P.ntiles = (int)n;
    int grid = std::max(1, std::min(grid_override ? grid_override : 148, P.ntiles));
    P.tiles_per_cta = (P.ntiles + grid - 1) / grid;
    grid = (P.ntiles + P.tiles_per_cta - 1) / P.tiles_per_cta;
    if (!warps) warps = 4;
    const int gwarps = std::max(1, std::min(warps, AMPO_GWARPS));
    std::vector<unsigned char> smem(amp::smem_bytes_ont(P.wt, warps, gwarps) + 64);
    unsigned char* sbase = smem.data();
    sbase += (16 - ((uintptr_t)sbase & 15)) & 15;
    P.gcap = P.tiles_per_cta;
    std::vector<uint32_t> glist((size_t)grid * P.gcap + 1);
    P.glist = glist.data();
    OntLaunch v{&P, sbase, mode, gwarps};
    for (int b = 0; b < grid; ++b) run_cta(b, warps * 32, ont_body, &v);
    return 0;
}

void emu_v7_stats(long long* out, int reset) {
    out[0] = amp::g_v7_stats[0]; out[1] = amp::g_v7_stats[1];
    if (reset) amp::g_v7_stats[0] = amp::g_v7_stats[1] = 0;
}

void emu_counts(void* h, int sample, int32_t* out) {
    EmuCtx* c = (EmuCtx*)h;
    for (int ch = 0; ch < AMP_NCH; ++ch)
        memcpy(out + (size_t)ch * c->L, c->counts.data() + ((size_t)sample * AMP_NCH + ch) * c->Lpad, (size_t)c->L * 4);
}
int* emu_counts_ptr(void* h) { return ((EmuCtx*)h)->counts.data(); }
int emu_lpad(void* h) { return ((EmuCtx*)h)->Lpad; }
long long emu_ins_count(void* h) { return (long long)((EmuCtx*)h)->cursor[1]; }
long long emu_ins_chars(void* h) {   // as amp_ins_count: a failed reservation leaves cursor[0] past the arena
    EmuCtx* c = (EmuCtx*)h;
    return (long long)std::min(c->cursor[0], c->tab.arena_words) * 8;
}
void emu_ins_export(void* h, int32_t* sample, int32_t* pos, int32_t* count, int64_t* str_off, char* chars) {
    EmuCtx* c = (EmuCtx*)h;
    int64_t o = 0; str_off[0] = 0;
    for (unsigned long long k = 0; k < c->cursor[1]; ++k) {
        const amp::InsSlot& s = c->slots[c->entries[k]];
        const unsigned char* rec = c->arena.data() + (s.key & 0xFFFFFFFFFFULL) * 8;
        int gpos; unsigned len; memcpy(&gpos, rec, 4); memcpy(&len, rec + 4, 4);
        sample[k] = gpos / c->Lpad; pos[k] = gpos % c->Lpad; count[k] = s.count;
        memcpy(chars + o, rec + 8, len); o += len; str_off[k + 1] = o;
    }
}
struct RawText {
    const char* p;
    char operator()(int i) const { return p[i]; }
    uint32_t word(int i, int len) const {
        uint32_t w = 0;
        for (int j = 0; j < 4 && i + j < len; ++j) w |= (uint32_t)(unsigned char)p[i + j] << (8 * j);
        return w;
    }
};
// the 64-bit hash ins_table_add computes for the key text[0, len) at gpos (home slot h & mask, tag (h >> 40) | 0x800000)
unsigned long long emu_ins_hash(int gpos, const char* text, int len) {
    const RawText t{text};
    unsigned long long h = amp::ins_hash_init(gpos);
    for (int i = 0; i < len; i += 4) h = amp::ins_hash_word(h, t.word(i, len));
    return amp::ins_hash_final(h, len);
}
void emu_ins_merge(void* h, long long n, const int32_t* sample, const int32_t* pos, const int32_t* count, const int64_t* str_off,
                   const char* chars) {
    EmuCtx* c = (EmuCtx*)h;
    for (long long k = 0; k < n; ++k) {
        RawText t{chars + str_off[k]};
        amp::ins_table_add(c->tab, sample[k] * c->Lpad + pos[k], (int)(str_off[k + 1] - str_off[k]), t, count[k]);
    }
}

// unit hooks for the sliding-window closed forms (q must have 8 readable bytes before and 16 after it for mode 2)
int emu_window(const uint8_t* q, int len, int W, int minq, int rev, int mode) {
    if (mode == 2) return amp::window_del_len_w4(q, len, minq, rev != 0);
    return rev ? amp::window_del_len_rev(q, len, W, minq) : amp::window_del_len_fwd(q, len, W, minq);
}

// unit hook: the register form of the [S]M[S] classification against the array form (returns 1 when they agree)
int emu_classify_agree(const uint32_t* cig, int nc, int l_seq) {
    amp::SimpleRead a, b;
    a.s1 = a.m = a.s2 = 0; a.mop = 0; b = a;
    const bool ra = amp::classify_simple(cig, nc, l_seq, a);
    const bool rb = amp::classify_simple3(nc, nc > 0 ? cig[0] : 0u, nc > 1 ? cig[1] : 0u, nc > 2 ? cig[2] : 0u, l_seq, b);
    if (ra != rb) return 0;
    return !ra || (a.s1 == b.s1 && a.m == b.m && a.s2 == b.s2 && a.mop == b.mop);
}

void emu_call(void* h, const char* ref_seq, int mdc, double mfc, int mdv, double mfv, int32_t* depth, int32_t* top_id,
              int32_t* top_count, uint8_t* pos_flags, int32_t* ref_count, double* fixed_freq, int32_t* fixed_rank,
              uint8_t* alt_mask, double* ins_freq, int32_t* ins_rank, uint8_t* ins_alt) {
    EmuCtx* c = (EmuCtx*)h;
    std::vector<int> heads((size_t)c->n_samples * c->Lpad, -1);
    for (unsigned long long k = 0; k < c->cursor[1]; ++k) {   // amp_link_kernel
        unsigned int s = c->entries[k];
        const unsigned char* rec = c->arena.data() + (c->slots[s].key & 0xFFFFFFFFFFULL) * 8;
        int gpos; memcpy(&gpos, rec, 4);
        c->slots[s].next = heads[gpos]; heads[gpos] = (int)s;
    }
    amp::CallParams P{};
    P.L = c->L; P.Lpad = c->Lpad; P.n_samples = c->n_samples; P.counts = c->counts.data(); P.slots = c->slots.data();
    P.slot_entry = c->slot_entry.data(); P.arena = c->arena.data(); P.heads = heads.data(); P.ref_seq = (const unsigned char*)ref_seq;
    P.min_depth_consensus = mdc; P.min_freq_consensus = mfc; P.min_depth_variants = mdv; P.min_freq_variants = mfv;
    P.depth = depth; P.top_id = top_id; P.top_count = top_count; P.pos_flags = pos_flags; P.ref_count = ref_count;
    P.fixed_freq = fixed_freq; P.fixed_rank = fixed_rank; P.alt_mask = alt_mask; P.ins_freq = ins_freq; P.ins_rank = ins_rank;
    P.ins_alt = ins_alt;
    static const unsigned char syms[8] = {'A', 'C', 'G', 'T', 'N', '-', 0, 0};
    for (long long gp = 0; gp < (long long)c->n_samples * c->L; ++gp) amp::call_position(P, syms, gp);
}


// ---- BGZF / BAM decode kernels (amp_bgzf.cuh): one warp of fibers per BGZF block ------------------------------------------------
struct InflateJob { const uint8_t* in; long long in_len; uint8_t* out; long long out_len; amp::InflateMem* mem; int err; };
static void inflate_body(void* a) {
    InflateJob* j = (InflateJob*)a;
    const int e = amp::inflate_block(j->in, j->in_len, j->out, j->out_len, *j->mem, amp::c_tid() & 31);
    if ((amp::c_tid() & 31) == 0) j->err = e;
}
// raw deflate stream -> out; returns the AMPZ_E_* bits
int emu_inflate(const uint8_t* in, long long in_len, uint8_t* out, long long out_len) {
    amp::InflateMem mem;
    InflateJob j{in, in_len, out, out_len, &mem, 0};
    run_cta(0, 32, inflate_body, &j);
    return j.err;
}
// BAM records of raw[lo, hi) (block-aligned chain) -> totals; returns 0 when the chain is not aligned
int emu_bam_totals(const uint8_t* raw, long long lo, long long hi, unsigned long long* out4) {
    amp::BamBlockTotals t;
    const bool ok = amp::bam_chain_totals(raw, lo, hi, t);
    out4[0] = t.n_rec; out4[1] = t.n_cig; out4[2] = t.n_seq; out4[3] = t.n_qual;
    return ok ? 1 : 0;
}
struct ScatterJob { const uint8_t* raw; long long lo, hi; amp::BamSoa D; };
static void scatter_body(void* a) {
    ScatterJob* j = (ScatterJob*)a;
    amp::bam_scatter_block(j->raw, j->lo, j->hi, j->D, 0, 0, 0, 0, amp::c_tid() & 31);
}
void emu_bam_scatter(const uint8_t* raw, long long lo, long long hi, int32_t* pos, uint16_t* flag, int32_t* tlen, uint32_t* cig_off,
                     uint32_t* cigar, uint32_t* seq_off, uint8_t* seq, uint32_t* qual_off, uint8_t* qual, unsigned long long* rec_off) {
    ScatterJob j{raw, lo, hi, amp::BamSoa{pos, flag, tlen, cig_off, cigar, seq_off, seq, qual_off, qual, rec_off}};
    run_cta(0, 32, scatter_body, &j);
}

// ---- trimmed BAM records rebuilt (amp_bgzf.cuh bam_rewrite_record): one warp of fibers, the selected records one after the other ----
struct RewriteJob { const uint8_t* raw; const unsigned long long* rec_off; const long long* sel; long long n_sel; const int32_t* new_pos;
                    const uint16_t* new_ncig; const uint32_t* cig_off; const uint32_t* new_cigar; uint8_t* out; long long total; };
static void rewrite_body(void* a) {
    RewriteJob* j = (RewriteJob*)a;
    const int lane = amp::c_tid() & 31;
    long long o = 0;
    for (long long k = 0; k < j->n_sel; ++k) {
        const long long i = j->sel[k];
        const uint32_t sz = amp::bam_new_record_size(j->raw, j->rec_off[i], j->new_ncig[i]);
        if (j->out) amp::bam_rewrite_record(j->raw, j->rec_off[i], j->new_pos[i], j->new_cigar + (size_t)j->cig_off[i] + 3 * (size_t)i, j->new_ncig[i], j->out + o, lane);
        o += sz;
        amp::w_sync();
    }
    if (lane == 0) j->total = o;
}
// same contract as amp_bam_rewrite of amp_hostio.cpp (out = NULL: size only)
long long emu_bam_rewrite(const uint8_t* raw, const unsigned long long* rec_off, const long long* sel, long long n_sel, const int32_t* new_pos,
                          const uint16_t* new_ncig, const uint32_t* cig_off, const uint32_t* new_cigar, uint8_t* out) {
    RewriteJob j{raw, rec_off, sel, n_sel, new_pos, new_ncig, cig_off, new_cigar, out, 0};
    run_cta(0, 32, rewrite_body, &j);
    return j.total;
}

// ---- BGZF deflate kernel (amp_deflate.cuh): one warp of fibers per block ------------------------------------------------------------
struct DeflateJob { const uint8_t* in; int n; uint32_t* out; int cap_words; amp::DeflateMem* mem; amp::DeflateTables* tab; int bytes; uint32_t crc; };
static void deflate_body(void* a) {
    DeflateJob* j = (DeflateJob*)a;
    const int lane = amp::c_tid() & 31;
    amp::deflate_tables_init(*j->tab, amp::c_tid(), amp::c_nthreads());
    amp::c_sync();
    const uint32_t mcol = amp::crc_shift_column(*j->tab, lane);
    static uint32_t tok[AMPD_SCRATCH];
    const int bytes = j->n >= 16 ? amp::deflate_block(j->in, j->n, *j->mem, *j->tab, j->out, j->cap_words, tok, lane) : -1;
    const uint32_t crc = amp::crc32_block(j->in, j->n, *j->tab, mcol, lane);
    if (lane == 0) { j->bytes = bytes; j->crc = crc; }
}
struct HuffJob { uint16_t* freq; int n; int maxlen; uint8_t* len; };
static void huff_body(void* a) {
    HuffJob* j = (HuffJob*)a;
    static uint32_t work[288]; static uint16_t order[288];
    amp::HuffWork W; W.a = work; W.order = order;
    amp::huff_lengths(j->freq, j->n, j->maxlen, j->len, W, amp::c_tid() & 31);
}
// code lengths of deflate_flush's code construction (freq may get two forced entries)
void emu_huff_lengths(uint16_t* freq, int n, int maxlen, uint8_t* len) {
    HuffJob j{freq, n, maxlen, len};
    run_cta(0, 32, huff_body, &j);
}
// in[0, n) (readable up to in + n + 8) -> raw deflate stream in out (cap_words 32-bit words + 64 words of slack); returns its length
// in bytes or -1 (does not fit / too short to bother); *crc = CRC-32 of the input
int emu_deflate(const uint8_t* in, int n, uint32_t* out, int cap_words, uint32_t* crc) {
    amp::DeflateMem mem; amp::DeflateTables tab;
    memset(&mem, 0xAB, sizeof mem); memset(&tab, 0xAB, sizeof tab);     // shared memory starts out with whatever the last kernel left
    DeflateJob j{in, n, out, cap_words, &mem, &tab, 0, 0};
    run_cta(0, 32, deflate_body, &j);
    *crc = j.crc;
    return j.bytes;
}

}  // extern "C"
