// amp_emu_call.cpp -- TEST INFRASTRUCTURE: the emulator of amp_emu.cpp plus the calling kernel's body (amp_call.cuh) on
// its fiber runtime, and insertion lists kept the way the device keeps them (ins_table_add links every allele it
// creates into InsTable.heads).  Not part of the product.
#include "amp_emu.cpp"
#include "../../amplipy_b200/csrc/amp_call.cuh"

#include <map>

static std::map<void*, std::vector<int>> g_heads;

struct CallLaunch { const amp::CallParams* P; const unsigned char* syms; long long n_pos; };
static void call_body(void* a) {
    CallLaunch* v = (CallLaunch*)a;
    const long long t = (long long)amp::c_block() * amp::c_nthreads() + amp::c_tid();
    if (t / AMP_CALL_LANES >= v->n_pos) return;
    amp::call_thread(*v->P, v->syms, t, amp::c_tid() & 31);
}

extern "C" {

// list heads for a fresh context (all -1): from here on ins_table_add links every allele it creates, as on the device
void emu_keep_lists(void* h) {
    EmuCtx* c = (EmuCtx*)h;
    std::vector<int>& v = g_heads[h];
    v.assign((size_t)c->n_samples * c->Lpad, -1);
    c->tab.heads = v.data();
}

// amp::call_thread with every CUDA thread a fiber, 256-thread CTAs as amp_call_device launches them, on the lists kept
// since emu_keep_lists (emu_call relinks the slots for its own lists: call this one first)
void emu_call_kernel(void* h, const char* ref_seq, int mdc, double mfc, int mdv, double mfv, int32_t* depth, int32_t* top_id,
                     int32_t* top_count, uint8_t* pos_flags, int32_t* ref_count, double* fixed_freq, int32_t* fixed_rank,
                     uint8_t* alt_mask, double* ins_freq, int32_t* ins_rank, uint8_t* ins_alt) {
    EmuCtx* c = (EmuCtx*)h;
    amp::CallParams P{};
    P.L = c->L; P.Lpad = c->Lpad; P.n_samples = c->n_samples; P.counts = c->counts.data(); P.slots = c->slots.data();
    P.slot_entry = c->slot_entry.data(); P.arena = c->arena.data(); P.heads = c->tab.heads; P.ref_seq = (const unsigned char*)ref_seq;
    P.min_depth_consensus = mdc; P.min_freq_consensus = mfc; P.min_depth_variants = mdv; P.min_freq_variants = mfv;
    P.depth = depth; P.top_id = top_id; P.top_count = top_count; P.pos_flags = pos_flags; P.ref_count = ref_count;
    P.fixed_freq = fixed_freq; P.fixed_rank = fixed_rank; P.alt_mask = alt_mask; P.ins_freq = ins_freq; P.ins_rank = ins_rank;
    P.ins_alt = ins_alt;
    static const unsigned char syms[8] = {'A', 'C', 'G', 'T', 'N', '-', 0, 0};
    CallLaunch v{&P, syms, (long long)c->n_samples * c->L};
    for (long long b = 0; b * 256 < v.n_pos * AMP_CALL_LANES; ++b) run_cta((int)b, 256, call_body, &v);
}

}  // extern "C"
