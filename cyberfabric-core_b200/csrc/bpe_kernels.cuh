// bpe_kernels.cuh -- the encode hot path as CUDA kernels for sm_100a.
//
//   K1  pretok_split_kernel (+ pretok_fixup_kernel)   packed prompt bytes -> piece-start bitmask      (SURVEY.md 8 a1)
//   K2s long_scan_kernel              finds the pieces longer than 32 bytes (work list of K2b / K2c), counts pieces per 2 KiB tile
//   K2a bpe_lookup_kernel             every short piece once: whole-piece lookup (CoreBPE's shortcut)       (a2)
//   K2m bpe_merge_kernel              the misses: exact min-rank merge loop, one lane per piece              (a2)
//   K2b bpe_long_kernel               pieces of 33.. bytes, one warp each: batched rounds + parallel-cut rounds (a2)
//   K2c bpe_list_kernel               the list phase of big pieces, one CTA each, state in shared memory     (a2)
//   K3  flag_count / tile_scan / emit_compact / prompt_offsets   token flags -> dense id stream + offsets + counts (a3, a4)
//   decode_len / decode_copy / decode_offsets                    ids -> bytes (SURVEY.md 8(f) item 2)
//
// Pure integer/indexing work: no tensor cores (north_star).  Bounds: HBM for the byte and id
// streams, L2 latency for the rank-table lookups (DESIGN.md section 4).
//
// The file compiles for the GPU with nvcc and, unchanged, for the CPU SIMT emulator used by
// the non-GPU tests (tests/simt/cusim.h defines the CUDA builtins); there is no CPU fallback
// in the product library.
#pragma once
#include <stdint.h>

#include "pretok.cuh"
#include "pretok_fsm.h"
#include "pretok_sync.cuh"
#include "tables.h"
#include "tma.cuh"

namespace cfbpe {

#ifdef CUSIM_EMULATOR
#define CFBPE_DYN_SMEM(name) uint32_t* const name = reinterpret_cast<uint32_t*>(cusim::dyn_smem())
#else
#define CFBPE_DYN_SMEM(name) extern __shared__ __align__(16) uint32_t name[]
#endif

constexpr uint32_t kMaxVocabs = 8;
// path counters for the emulator tests (which path did a test actually exercise); nothing on the device
#ifdef CUSIM_EMULATOR
inline unsigned long long* dbg_counters() { static unsigned long long c[16]; return c; }
#define CFBPE_DBG_COUNT(i) (++dbg_counters()[i])
#else
#define CFBPE_DBG_COUNT(i) ((void)0)
#endif
// 0: pieces deferred to bpe_list_kernel  1: list -> batched switches (medium pieces)  2: the same in bpe_list_kernel
// 3: K1 bulk whitespace runs  4: K1 bulk digit runs  5: pieces on the global-memory list path
// 6: rounds of bpe_list_kernel  7: merges taken in them
// 8: K1 calls of the per-character walker (a lane crossed its 32-byte window)  9: characters it walked  10: K1 warp tiles

#ifndef CFBPE_SPLIT_CHUNK
#define CFBPE_SPLIT_CHUNK 64
#endif
constexpr uint32_t kSplitChunk = CFBPE_SPLIT_CHUNK;     // bytes of text per K1 thread
constexpr uint32_t kBigPiece = 256;      // bytes: K2b serves longer pieces first (tail latency)
constexpr uint32_t kScanTileWords = 256;   // flag words per K3 tile (= 8 KiB of text); one word per thread

struct VocabSet {
    TablesView v[kMaxVocabs];      // slots that are not loaded alias a loaded one (a bad id from a device-path caller must not fault) ...
    uint32_t loaded_mask;          // ... and prompt_map_kernel reports it (DeviceStatus::bad_vocab)
};

struct BatchView {
    const uint8_t* bytes;      // packed prompt bytes (+ >= 16 bytes of readable padding)
    const uint64_t* offsets;   // n_prompts + 1
    const uint8_t* vocab_ids;  // n_prompts or nullptr
    uint32_t n_prompts;
    uint64_t total_bytes;
};

// status word written by the kernels
struct DeviceStatus {
    uint32_t bad_utf8;     // != 0: some prompt held malformed UTF-8
    uint32_t n_long;       // number of long pieces queued for K2b
    uint32_t long_overflow;
    uint32_t long_next;    // K2b work ticket (pieces of 33..kBigPiece bytes)
    uint32_t n_big;        // pieces longer than kBigPiece (stored from the back of the list)
    uint32_t defer_next;   // K2c work ticket (over the big pieces; those K2b deferred carry their part count)
    uint64_t n_tokens;     // ids produced by this (sub-)batch (written by tile_scan)
    uint64_t tok_end;      // token_base + n_tokens: where the next sub-batch of a pipelined call continues
    unsigned long long long_bytes;   // bytes inside pieces handled by K2b ...
    unsigned long long long_tokens;  // ... and the ids they became (for the roofline of that kernel)
    uint32_t miss_n[3];    // short pieces that are not one token, by length class: 13..32 | 7..12 | 2..6 bytes (K2a -> K2m)
    uint32_t miss_next[3]; // K2m work tickets
    uint32_t miss_overflow;
    uint32_t extra_n;      // tokens of merged short pieces written to DenseIds::extras so far
    uint32_t split_next;   // K1 work ticket: the next warp tile (tiles differ widely in cost: a tile that enters a 4 KiB run costs ten average ones)
    uint32_t fix_n;        // K1 threads that stopped in S_W_U (pretok_fixup_kernel finishes them)
    uint32_t bad_vocab;    // != 0: a prompt names a vocabulary id that is not loaded (device-path callers; the host paths check before)
    uint32_t defer_n;      // pieces K2b handed to K2c ...
    unsigned long long defer_parts;   // ... and their parts at hand-over
};

// K2a's lists of the short pieces that need the merge loop, one per length class (worst-case capacities: a class with
// pieces of >= L bytes holds at most total / L of them)
struct MissLists {
    uint64_t* list[3];     // byte position | rank of the piece << 32
    uint32_t cap[3];
};
__host__ __device__ inline uint32_t miss_class_min_len(uint32_t c) { return c == 0 ? 13u : (c == 1 ? 7u : 1u); }

struct LongPiece { uint64_t start; uint64_t end; uint32_t vocab; uint32_t pad; };   // pad: 0, or the part count K2b left for K2c

// ---------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------
// index of the prompt that contains byte position pos (pos < total): largest i with offsets[i] <= pos
__device__ __forceinline__ uint32_t find_prompt(const uint64_t* __restrict__ offsets, uint32_t n, uint64_t pos) {
    uint32_t lo = 0, hi = n;  // invariant: offsets[lo] <= pos < offsets[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= pos) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void or_bits(uint32_t* __restrict__ words, uint64_t word, uint32_t bits) {
    if (bits) atomicOr(&words[word], bits);
}

// L2 prefetch of the line at p (a long run is scanned by ONE lane: without it every iteration is a DRAM round trip)
__device__ __forceinline__ void prefetch_l2(const void* p) {
#if !defined(CUSIM_EMULATOR)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

// end of the run of bytes equal to c that starts at pos (pos < pe, s[pos] == c need not hold): first position in
// [pos, pe) whose byte differs, 16 bytes per load once aligned
__device__ __forceinline__ uint64_t same_byte_run_end(const uint8_t* __restrict__ s, uint64_t pos, uint64_t pe, uint32_t c) {
    uint64_t e = pos;
    while (e < pe && (reinterpret_cast<uintptr_t>(s + e) & 15u)) { if (s[e] != c) return e; ++e; }
    const uint32_t w = c * 0x01010101u;
    for (uint64_t a = e; a < pe && a < e + 1024; a += 128) prefetch_l2(s + a);
    while (e + 128 <= pe) {     // eight loads in flight: the loop is one dependent memory round trip per iteration
        if (e + 1024 < pe) prefetch_l2(s + e + 1024);
        uint4 v[8];
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) v[k] = *reinterpret_cast<const uint4*>(s + e + 16 * k);
        uint32_t d = 0;
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) d |= (v[k].x ^ w) | (v[k].y ^ w) | (v[k].z ^ w) | (v[k].w ^ w);
        if (d) break;
        e += 128;
    }
    while (e + 16 <= pe) {
        const uint4 v = *reinterpret_cast<const uint4*>(s + e);
        if (v.x != w || v.y != w || v.z != w || v.w != w) break;
        e += 16;
    }
    while (e < pe && s[e] == c) ++e;
    return e;
}
__device__ __forceinline__ bool four_ascii_digits(uint32_t w) {
    const uint32_t t = w ^ 0x30303030u;                       // a digit byte becomes 0..9
    return ((((t & 0x7F7F7F7Fu) + 0x76767676u) | t) & 0x80808080u) == 0u;
}
__device__ __forceinline__ uint64_t ascii_digit_run_end(const uint8_t* __restrict__ s, uint64_t pos, uint64_t pe) {
    uint64_t e = pos;
    while (e < pe && (reinterpret_cast<uintptr_t>(s + e) & 15u)) { if ((s[e] - '0') >= 10u) return e; ++e; }
    for (uint64_t a = e; a < pe && a < e + 1024; a += 128) prefetch_l2(s + a);
    while (e + 128 <= pe) {      // eight loads in flight (see same_byte_run_end)
        if (e + 1024 < pe) prefetch_l2(s + e + 1024);
        uint4 v[8];
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) v[k] = *reinterpret_cast<const uint4*>(s + e + 16 * k);
        bool ok = true;
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) ok = ok && four_ascii_digits(v[k].x) && four_ascii_digits(v[k].y) && four_ascii_digits(v[k].z) && four_ascii_digits(v[k].w);
        if (!ok) break;
        e += 128;
    }
    while (e + 16 <= pe) {
        const uint4 v = *reinterpret_cast<const uint4*>(s + e);
        if (!(four_ascii_digits(v.x) && four_ascii_digits(v.y) && four_ascii_digits(v.z) && four_ascii_digits(v.w))) break;
        e += 16;
    }
    while (e < pe && (s[e] - '0') < 10u) ++e;
    return e;
}

// ---------------------------------------------------------------------------------------
// K1: pre-tokenizer split.  One thread per kSplitChunk bytes.  A thread starts at the first sync
// point of its chunk (prompt start or is_sync_point) and runs the table-driven automaton of
// pretok_fsm.h, ONE CHARACTER PER ITERATION, until it stands on a sync point at or beyond the end
// of its chunk -- which is where a later thread started.  All lanes execute the same instruction
// stream whatever match they are in (the first version walked whole matches per thread: 4.3 of 32
// lanes active, profiles/ncu_lines_pretok_split_r01a.txt).
// ---------------------------------------------------------------------------------------
// A thread that started in S_W_U (pretok_sync.cuh) and meets an upper-case letter needs the automaton's real state.  Finding
// it is a look-back of unbounded length: inlined -- or even called -- in the hot loop it cost the kernel registers and 17 %
// of its speed, so the thread files the position and stops, and pretok_fixup_kernel (next launch, almost always empty)
// finds the state and finishes that thread's job.
struct SplitFix { uint32_t pos, ce; };   // byte positions inside the (sub-)batch (< 4 GiB): where to resume, and from where on the walker may hand over

// kMode 0: the thread of chunk [cs, ce) (first form of K1: one thread per 64 bytes).
// kMode 1: resume at fix_pos on behalf of a walker that stopped in an undecided state; the real state is found by looking back.
// kMode 2: resume at fix_pos with the state and remembered positions a lane of pretok_split16_kernel hands over (long runs).
// kRow / kTabSize: row stride and size per pattern of the transition table at s_fsm (12-wide in the first form, 16-wide in K1 v2).
template <int kMode, uint32_t kRow = X_COUNT, uint32_t kTabSize = kPretokTableSize>
__device__ __forceinline__ void split_thread(const BatchView& b, const VocabSet& vs, UcTables uc, const uint16_t* s_fsm, const uint8_t* s_ascii,
                                             uint32_t* __restrict__ piece_bits, DeviceStatus* status, SplitFix* fix_list, uint32_t fix_cap,
                                             uint64_t cs, uint64_t ce, uint64_t fix_pos, uint32_t fix_pidx,
                                             uint32_t state2 = 0, uint64_t alc2 = 0, uint64_t last2 = 0, uint64_t lbe2 = 0, uint32_t pats2 = 0) {
    constexpr bool kFix = kMode != 0;       // resumed walkers mark with atomics and never search for a sync point
    // (mode 2 gets the pattern ids of the vocabulary slots packed four bits each: a VocabSet passed down an out-of-line call would
    //  be copied to the stack)
    auto pat_of = [&](uint32_t p) -> uint32_t {
        const uint32_t v = b.vocab_ids ? b.vocab_ids[p] : 0u;
        return kMode == 2 ? ((pats2 >> (4u * (v & 7u))) & 15u) : vs.v[v].pattern_id;
    };
    // (a shared-memory text tile with coalesced 16-byte loads was measured slower here: occupancy fell from 67 % to
    //  29 % and the accessor cost more than the L1 hits it replaced -- profiles/ncu_summary_r01k.json)
    const uint8_t* __restrict__ s = b.bytes;

    // (a resumed walker has consumed at least one byte of the prompt it is in: fix_pos may be that prompt's END)
    uint32_t pidx = kFix ? (fix_pidx != 0xFFFFFFFFu ? fix_pidx : find_prompt(b.offsets, b.n_prompts, fix_pos - 1)) : find_prompt(b.offsets, b.n_prompts, cs);
    uint64_t ps = b.offsets[pidx], pe = b.offsets[pidx + 1];
    uc.ascii_x = s_ascii;   // the copy in shared memory

    // ---- find the first sync point in [cs, ce)
    uint64_t pos = kFix ? fix_pos : cs;
    uint32_t state = kNoSync;
    uint32_t prevx = X_EOT, nlet = 0, npun = 0;   // class of the previous character; consecutive letters (<= 3) / punctuation (<= 2) before pos
    uint32_t pat = pat_of(pidx);
    uint64_t lbe_fix = 0;
    if (kMode == 1) {   // the real state at fix_pos (inside a prompt, after a letter), and the classes the hand-over looks at
        sync_state(s, pos, ps, pe, uc, true, &prevx, &nlet, &npun);
        state = resolve_word_state<kRow>(s, pos, ps, pe, uc, s_fsm + pat * kTabSize, &lbe_fix);
    }
#ifdef CUSIM_EMULATOR
    if (kMode == 1 && getenv("CFBPE_DBG")) fprintf(stderr, "fixup: pos %llu ce %llu state %u lbe %llu pidx %u ps %llu pe %llu\n", (unsigned long long)pos, (unsigned long long)ce, state, (unsigned long long)lbe_fix, pidx, (unsigned long long)ps, (unsigned long long)pe);
#endif
    if (kMode == 2) {   // state handed over; the classes of the last three characters from memory
        if (pos < pe) sync_state(s, pos, ps, pe, uc, (pat & 1u) != 0, &prevx, &nlet, &npun);
        state = state2; lbe_fix = lbe2;
    }
    while (!kFix && pos < ce) {
        if (pos == pe) {  // step into the next non-empty prompt
            do { ++pidx; ps = pe; pe = b.offsets[pidx + 1]; } while (pe == ps);
            pat = pat_of(pidx);
        }
        prevx = X_EOT; nlet = 0; npun = 0;
        state = (pos == ps) ? static_cast<uint32_t>(S_START) : sync_state(s, pos, ps, pe, uc, (pat & 1u) != 0, &prevx, &nlet, &npun);
        if (state != kNoSync) break;
        ++pos;
    }
    if (state == kNoSync) return;

    // ---- run the automaton
    const uint16_t* tab = s_fsm + pat * kTabSize;
    uint64_t alc = kMode == 2 ? alc2 : 0, last = kMode == 2 ? last2 : 0, lbe = kFix ? lbe_fix : pos;     // (lbe = pos: what W_XB0 would hold if that is what S_W_U turns out to be)
    int bad = 0;
    // boundaries inside my chunk collect in one 64-bit mask (the chunk is 64-byte aligned: two flag words, OR-ed in at the
    // end because the thread to my left may have set bits there while handing over); those beyond it go out one by one
    static_assert(kSplitChunk <= 64, "the chunk mask is one 64-bit word");
    uint64_t mine = 0;
    auto mark = [&](uint64_t p) {
        if (!kFix && p - cs < kSplitChunk) mine |= 1ull << (p - cs);
        else atomicOr(&piece_bits[p >> 5], 1u << (p & 31));
    };
#ifdef CUSIM_EMULATOR
    const uint64_t dbg_pos0 = pos; uint64_t dbg_iters = 0;
    struct DbgWalk { uint64_t p0, *it, *pp; const uint8_t* s; int mode; ~DbgWalk() { if (getenv("CFBPE_DBG_WALK") && *it > (uint64_t)atoi(getenv("CFBPE_DBG_WALK"))) { fprintf(stderr, "walk mode %d: %llu iterations from %llu to %llu: ", mode, (unsigned long long)*it, (unsigned long long)p0, (unsigned long long)*pp); for (int i = 0; i < 40; ++i) fputc(s[p0 + i] >= 32 && s[p0 + i] < 127 ? s[p0 + i] : '.', stderr); fputc('\n', stderr); } } } dbg_walk{dbg_pos0, &dbg_iters, &pos, s, kMode};
#endif
    if (kMode == 2) CFBPE_DBG_COUNT(8);
#if defined(CFBPE_TILE_CLOCK) && !defined(CUSIM_EMULATOR)
    const long long rs_t0 = clock64(); long long rs_bulk = 0, rs_scan = 0; unsigned rs_iters = 0; const uint64_t rs_pos0 = pos;
    struct RsPrint { const long long* t0; long long* bulk; long long* scan; unsigned* it; const uint64_t* p0; const uint64_t* p1; int mode;
        __device__ ~RsPrint() { const long long dt = clock64() - *t0; if (mode == 2 && dt > 40000) printf("  resume: %lld cycles, %u iterations, bulk %lld (scan %lld), %llu bytes from %llu\n", dt, *it, *bulk, *scan, (unsigned long long)(*p1 - *p0), (unsigned long long)*p0); } } rs_print{&rs_t0, &rs_bulk, &rs_scan, &rs_iters, &rs_pos0, &pos, kMode};
#endif
    for (;;) {
#if defined(CFBPE_TILE_CLOCK) && !defined(CUSIM_EMULATOR)
        ++rs_iters;
#endif
#ifdef CUSIM_EMULATOR
        ++dbg_iters;
        if (kMode == 2) CFBPE_DBG_COUNT(9);
#endif
        uint32_t x, len, b0 = 0x100u;
        if (pos == pe) { x = X_EOT; len = 0; }
        else {
            b0 = s[pos];
            if (b0 < 0x80) { x = s_ascii[b0]; len = 1; }
            else { const Ch c = get_char(s, pos, pe, uc, &bad); x = c.cls; len = c.len; }
        }
        uint32_t a = tab[state * kRow + x];
        if (kMode != 1 && (a & A_RESOLVE)) {   // started inside a run of both-sets / upper-case letters, and now it matters what came before it
            const uint32_t k = atomicAdd(&status->fix_n, 1u);
            if (k < fix_cap) { SplitFix f; f.pos = static_cast<uint32_t>(pos); f.ce = static_cast<uint32_t>(ce); fix_list[k] = f; }
            else atomicOr(&status->long_overflow, 1u);
            break;
        }
        uint32_t skip = 0;
        if (a & A_CONTR) {
            skip = contraction_bytes(s, pos, pe);
            if (skip && (a & A_CONTR_SUFFIX)) a &= ~A_B_NOW;   // the contraction belongs to the piece that just ended
        }
        // retroactive boundaries (all at positions I own)
        if (a & (A_EMIT_ALC | A_EMIT_LAST | A_EMIT_LBE)) {
            if (a & A_EMIT_ALC) mark(alc);
            if (a & A_EMIT_LAST) mark(last);
            if (a & A_EMIT_LBE) mark(lbe);
        }
        if (x == X_EOT) {
            if (pos >= b.total_bytes) break;
            do { ++pidx; ps = pe; pe = b.offsets[pidx + 1]; } while (pe == ps);
            if (pos >= ce) break;            // the next prompt's first byte is a sync point of a later chunk
            pat = pat_of(pidx);
            tab = s_fsm + pat * kTabSize;
            state = S_START;
            prevx = X_EOT; nlet = 0; npun = 0;
            continue;
        }
        // hand over to the thread that started at the first sync point at or beyond the end of my chunk
        // (after the retroactive boundaries above, which concern positions of mine); same predicate as
        // sync_state(), evaluated on the classes just seen
        if (pos >= ce && (bad || sync_rule(x, prevx, nlet, npun, (pat & 1u) != 0) != kNoSync)) break;
        if (a & A_B_NOW) mark(pos);
        if (a & A_SET_ALC) alc = pos + len;
        if (a & A_SET_LAST) last = pos;
        if (a & A_SET_LBE) lbe = pos + len;
        // the hand-over predicate needs the classes of the last three characters only once pos reaches ce: track them
        // from 16 bytes (>= 4 characters) before that, so that the counters are exact when they are first read
        const bool track = pos + 16 >= ce;
        if (skip) {   // a contraction: apostrophe + one or two letters
            state = S_START; pos += skip;
            if (track) {
                const uint32_t lb = s[pos - 1];
                prevx = lb < 0x80 ? s_ascii[lb] : static_cast<uint32_t>(X_LL);   // last letter of the contraction (U+017F is Ll)
                nlet = (skip == 3 && lb >= 0x80) ? 1u : skip - 1;
                npun = 0;
            }
        } else {
            state = a & A_STATE_MASK; pos += len;
            if (track) {
                prevx = x;
                nlet = x_is_letter(x) ? (nlet < 3 ? nlet + 1 : 3u) : 0u;
                npun = x_is_run_punct(x, (pat & 1u) != 0) ? (npun < 2 ? npun + 1 : 2u) : 0u;
            } else { nlet = 0; npun = 0; }
            // ---- runs that hold no sync point -- one whitespace byte repeated, ASCII digits -- are taken in bulk: the one
            //      thread that entered such a run would otherwise walk it a character per iteration (~200 cycles each,
            //      nothing else to hide the latency) while the rest of the grid has long finished.  Only beyond the end of
            //      my chunk: inside it the walk is bounded anyway, and short runs (indentation, years) are cheaper per character
#if defined(CFBPE_TILE_CLOCK) && !defined(CUSIM_EMULATOR)
            const long long rs_b0 = clock64();
#endif
            if (pos >= ce && b0 < 0x80u && pos < pe) {
                if ((x == X_SPACE || x == X_CRLF || x == X_WS) && s[pos] == b0) {
                    const uint32_t a2 = tab[state * kRow + x];
                    if ((a2 & A_STATE_MASK) == state && !(a2 & (A_B_NOW | A_EMIT_ALC | A_EMIT_LAST | A_EMIT_LBE | A_CONTR))) {
                        CFBPE_DBG_COUNT(3);
                        const uint64_t e = same_byte_run_end(s, pos, pe, b0);    // self-loop: only the remembered positions move
                        if (a2 & A_SET_ALC) alc = e;
                        if (a2 & A_SET_LAST) last = e - 1;
                        if (a2 & A_SET_LBE) lbe = e;
                        pos = e; prevx = x; nlet = 0; npun = 0;
                    }
                } else if (x == X_N && state >= S_D1 && state <= S_D3 && (s[pos] - '0') < 10u) {
                    // \p{N}{1,md}: a boundary every md digits, counted from the start of the run
                    const uint32_t md = (tab[S_D1 * kRow + X_N] & A_B_NOW) ? 1u : ((tab[S_D2 * kRow + X_N] & A_B_NOW) ? 2u : 3u);
                    CFBPE_DBG_COUNT(4);
                    const uint64_t e = ascii_digit_run_end(s, pos, pe);
#if defined(CFBPE_TILE_CLOCK) && !defined(CUSIM_EMULATOR)
                    rs_scan += clock64() - rs_b0;
#endif
                    const uint32_t d = state - S_D1 + 1u;                        // digits in the current piece so far
                    {   // a boundary every md digits from `first` on: one flag word at a time (the pattern repeats: a loop over
                        // the boundaries took 200 cycles each, 100 000 for a run of 1.4 KiB -- profiles/k1_tiles_r02.txt)
                        const uint64_t first = pos + (md - d);
                        const uint32_t pat_bits = md == 1u ? 0xFFFFFFFFu : (md == 2u ? 0x55555555u : 0x49249249u);
                        if (first < e) {
                            uint32_t off = static_cast<uint32_t>(first & 31u);          // first boundary of the word, as a bit index
                            const uint32_t adv = 4u % md;                               // 36 = 0 (mod 1, 2, 3): the offset moves by (36 - 32) mod md a word
                            for (uint64_t w = first >> 5; w <= (e - 1) >> 5; ++w) {
                                const uint64_t w0 = w << 5;
                                uint32_t m = pat_bits << off;
                                if (e < w0 + 32u) m &= (1u << static_cast<uint32_t>(e - w0)) - 1u;
                                if (m) atomicOr(&piece_bits[w], m);
                                off = off % md + adv; if (off >= md) off -= md;
                            }
                        }
                    }
                    state = S_D1 + static_cast<uint32_t>((d - 1u + (e - pos)) % md);
                    pos = e; prevx = X_N; nlet = 0; npun = 0;
                }
            }
#if defined(CFBPE_TILE_CLOCK) && !defined(CUSIM_EMULATOR)
            rs_bulk += clock64() - rs_b0;
#endif
        }
    }
    if (!kFix) {
        or_bits(piece_bits, cs >> 5, static_cast<uint32_t>(mine));
        or_bits(piece_bits, (cs >> 5) + 1, static_cast<uint32_t>(mine >> 32));
    }
    if (bad) atomicOr(&status->bad_utf8, 1u);
}

__global__ void __launch_bounds__(256)
pretok_split_kernel(BatchView b, VocabSet vs, UcTables uc, uint32_t* __restrict__ piece_bits, DeviceStatus* status, SplitFix* fix_list, uint32_t fix_cap) {
    __shared__ uint16_t s_fsm[kNumPatterns * kPretokTableSize];
    __shared__ uint8_t s_ascii[128];
    for (uint32_t i = threadIdx.x; i < kNumPatterns * kPretokTableSize; i += blockDim.x) s_fsm[i] = uc.fsm[i];
    if (threadIdx.x < 128) s_ascii[threadIdx.x] = uc.ascii_x[threadIdx.x];
    __syncthreads();
    const uint64_t chunk = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const uint64_t cs = chunk * kSplitChunk;
    if (cs >= b.total_bytes) return;
    const uint64_t ce = (cs + kSplitChunk < b.total_bytes) ? cs + kSplitChunk : b.total_bytes;
    split_thread<0>(b, vs, uc, s_fsm, s_ascii, piece_bits, status, fix_list, fix_cap, cs, ce, 0, 0);
}

// the threads of pretok_split_kernel that stopped in S_W_U at an upper-case letter: one thread each (grid-stride)
__global__ void __launch_bounds__(256)
pretok_fixup_kernel(BatchView b, VocabSet vs, UcTables uc, uint32_t* __restrict__ piece_bits, DeviceStatus* status, const SplitFix* fix_list, uint32_t fix_cap) {
    __shared__ uint16_t s_fsm[kNumPatterns * kPretokTableSize];
    __shared__ uint8_t s_ascii[128];
    const uint32_t n = status->fix_n < fix_cap ? status->fix_n : fix_cap;
    if (blockIdx.x * blockDim.x >= n) return;          // nothing filed: the usual case
    for (uint32_t i = threadIdx.x; i < kNumPatterns * kPretokTableSize; i += blockDim.x) s_fsm[i] = uc.fsm[i];
    if (threadIdx.x < 128) s_ascii[threadIdx.x] = uc.ascii_x[threadIdx.x];
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const SplitFix f = fix_list[i];
        split_thread<1>(b, vs, uc, s_fsm, s_ascii, piece_bits, status, nullptr, 0, 0, f.ce, f.pos, 0xFFFFFFFFu);
    }
}


constexpr uint32_t kFull = 0xFFFFFFFFu;
// ---------------------------------------------------------------------------------------
// bit helpers shared by the K2 kernels
// ---------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t lanemask_lt(uint32_t lane) { return (1u << lane) - 1u; }

// 33 piece-start bits for positions ws .. ws+32 (bit i <-> ws+i); words beyond n_words read as 0
__device__ __forceinline__ uint64_t load_bits33(const uint32_t* __restrict__ bits, uint64_t n_words, uint64_t ws) {
    const uint64_t w = ws >> 5;
    const uint32_t sh = static_cast<uint32_t>(ws & 31);
    const uint64_t lo = bits[w];
    const uint64_t hi = (w + 1 < n_words) ? bits[w + 1] : 0;
    const uint64_t v = (lo | (hi << 32)) >> sh;   // 64 - sh >= 33 valid bits
    return v & 0x1FFFFFFFFull;
}

// next set bit at position >= from and < limit in the bit array, or limit
__device__ __forceinline__ uint64_t next_set_bit(const uint32_t* __restrict__ bits, uint64_t from, uint64_t limit) {
    if (from >= limit) return limit;
    uint64_t w = from >> 5;
    uint32_t cur = bits[w] & (kFull << (from & 31));
    const uint64_t wl = (limit + 31) >> 5;
    while (!cur) {
        if (++w >= wl) return limit;
        cur = bits[w];
    }
    const uint64_t p = (w << 5) + (__ffs(cur) - 1);
    return p < limit ? p : limit;
}


// ---------------------------------------------------------------------------------------
// K2 (lane-per-piece form).  The window kernel above spends ~19 warp-instructions per byte because one
// lane per BYTE executes the whole-piece lookup and every merge round, while only the head lane of each
// piece does useful work in the lookup, and a round advances one merge per piece (ncu: profiles/).  Here a
// lane owns PIECES:
//   pass 1  each lane walks the pieces that start in its 16 bytes of the warp's 512-byte range and does
//           CoreBPE's whole-piece lookup (short table: key = the piece's <= 12 bytes; long table: hash + verify).
//           Hits are final.  Pieces longer than 32 bytes go to the K2b work list.
//   pass 2  the misses of the whole warp are dealt out densely, 32 at a time, one piece per lane; each lane
//           runs the exact sequential merge loop on its piece with the parts in shared memory
//           (tiktoken/_educational.py:95-110: leftmost minimum rank, until no adjacent pair is a token).
// ---------------------------------------------------------------------------------------
constexpr uint32_t kPieceRange = 512;     // bytes of text per warp: 16 per lane
constexpr uint32_t kPieceWarps = 4;       // warps per CTA

// bytes [p, p+16) as four little-endian words, read with aligned 32-bit loads (p may be unaligned; the buffer is
// readable up to 16 bytes past the last prompt byte)
__device__ __forceinline__ void load16(const uint8_t* __restrict__ p, uint32_t& w0, uint32_t& w1, uint32_t& w2, uint32_t& w3) {
    const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
    const uint32_t* q = reinterpret_cast<const uint32_t*>(addr & ~static_cast<uintptr_t>(3));
    const uint32_t sh = static_cast<uint32_t>(addr & 3) * 8;
    const uint32_t a = q[0], bq = q[1], c = q[2], d = q[3];
    if (sh == 0) { w0 = a; w1 = bq; w2 = c; w3 = d; }
    else {
        const uint32_t e = q[4];
        w0 = __funnelshift_r(a, bq, sh); w1 = __funnelshift_r(bq, c, sh); w2 = __funnelshift_r(c, d, sh); w3 = __funnelshift_r(d, e, sh);
    }
}

// CoreBPE's `if piece in ranks` for a piece of 1..32 bytes at p
__device__ __forceinline__ uint32_t whole_piece_lookup(const TablesView& T, const uint8_t* __restrict__ p, uint32_t len) {
    if (len > T.max_token_len) return kNone;
    // (a separate path for pieces of <= 4 bytes -- two words loaded instead of five, a two-byte piece as a direct index into the
    //  byte-pair table -- made K2a 13 % SLOWER: the lanes of a warp then run two paths one after the other; profiles/bench_r02w.json)
    uint32_t w0, w1, w2, w3;
    load16(p, w0, w1, w2, w3);
    uint64_t k0 = static_cast<uint64_t>(w0) | (static_cast<uint64_t>(w1) << 32);
    uint32_t k1 = w2;
    if (len < 8) k0 &= (1ull << (8 * len)) - 1ull;
    if (len <= 8) k1 = 0; else if (len < 12) k1 &= (1u << (8 * (len - 8))) - 1u;
    if (len <= kShortMaxLen) return short_lookup(T, k0, k1, len);
    return long_lookup(T, long_hash(k0, k1, load_le32(p + len - 4), len), p, len);
}

// the exact merge loop on one piece of 2..32 bytes.  Part k = the part that STARTS at byte k of the piece; `alive` has
// one bit per live part, so a merge clears a bit instead of shifting arrays.  Shared-memory columns (stride 32 words):
//   sid[k*32] = id of part k      srk[k*32] = rank of (part k, next live part)
__device__ __forceinline__ uint32_t merge_piece_in_lane(const TablesView& T, const uint8_t* __restrict__ text, uint64_t pos, uint32_t len,
                                                        uint32_t* sid, uint32_t* srk, uint32_t* __restrict__ tok_bits) {
    const uint8_t* __restrict__ p = text + pos;
    // the piece's bytes (<= 32) in eight registers; parts = bytes, ranks from the raw byte-pair table, four loads in flight
    uint32_t w[8];
    load16(p, w[0], w[1], w[2], w[3]);
    if (len > 16) load16(p + 16, w[4], w[5], w[6], w[7]); else { w[4] = w[5] = w[6] = w[7] = 0; }
    auto byte_at = [&](uint32_t k) -> uint32_t {   // k < 32; selects without dynamic register indexing
        const uint32_t lo4 = (k & 4u) ? ((k & 8u) ? ((k & 16u) ? w[7] : w[3]) : ((k & 16u) ? w[5] : w[1]))
                                       : ((k & 8u) ? ((k & 16u) ? w[6] : w[2]) : ((k & 16u) ? w[4] : w[0]));
        return (lo4 >> (8u * (k & 3u))) & 0xFFu;
    };
    for (uint32_t k0 = 0; k0 < len; k0 += 4) {
        uint32_t bv[5], idv[4], rkv[4];
#pragma unroll
        for (uint32_t t = 0; t < 5; ++t) bv[t] = (k0 + t < len) ? byte_at(k0 + t) : 0u;
#pragma unroll
        for (uint32_t t = 0; t < 4; ++t) {
            idv[t] = (k0 + t < len) ? T.byte2id[bv[t]] : 0u;
            rkv[t] = (k0 + t + 1 < len) ? T.bytepair[(bv[t] << 8) | bv[t + 1]] : kNone;
        }
#pragma unroll
        for (uint32_t t = 0; t < 4; ++t) if (k0 + t < len) { sid[(k0 + t) * 32] = idv[t]; srk[(k0 + t) * 32] = rkv[t] == kNone ? kNone : ((rkv[t] << 5) | (k0 + t)); }
    }
    uint32_t alive = (len >= 32) ? kFull : ((1u << len) - 1u);
    for (;;) {
        uint32_t bkey = kNone;
        for (uint32_t bits = alive; bits; bits &= bits - 1) {     // key = rank << 5 | position: the minimum is the leftmost minimum rank
            const uint32_t k = static_cast<uint32_t>(__ffs(bits)) - 1u;
            const uint32_t r = srk[k * 32];
            bkey = r < bkey ? r : bkey;
        }
        if (bkey == kNone) break;
        const uint32_t best = bkey >> 5, bi = bkey & 31u;
        const uint32_t above = alive & ~((2u << bi) - 1u);
        const uint32_t nb = static_cast<uint32_t>(__ffs(above)) - 1u;          // the partner: it has one, its rank was not kNone
        alive &= ~(1u << nb);
        sid[bi * 32] = best;                                                    // rank == id of the merged token
        const uint32_t above2 = alive & ~((2u << bi) - 1u);
        const uint32_t below = alive & ((1u << bi) - 1u);
        const bool wr = above2 != 0, wl = below != 0;
        const uint32_t nn = wr ? static_cast<uint32_t>(__ffs(above2)) - 1u : 0u;
        const uint32_t pv = wl ? 31u - static_cast<uint32_t>(__clz(below)) : 0u;
        uint32_t nr, nl;
        pair_lookup2(T, best, wr ? sid[nn * 32] : 0u, wr, wl ? sid[pv * 32] : 0u, best, wl, nr, nl);
        srk[bi * 32] = nr == kNone ? kNone : ((nr << 5) | bi);
        if (wl) srk[pv * 32] = nl == kNone ? kNone : ((nl << 5) | pv);
    }
    const uint64_t mask = static_cast<uint64_t>(alive) << (pos & 31);
    atomicOr(&tok_bits[pos >> 5], static_cast<uint32_t>(mask));
    if (mask >> 32) atomicOr(&tok_bits[(pos >> 5) + 1], static_cast<uint32_t>(mask >> 32));
    return alive;      // the ids of the live parts are in sid[k * 32]
}

__device__ __forceinline__ uint32_t kth_set_bit(uint32_t mask, uint32_t k) {   // position of the k-th (0-based) set bit
    for (uint32_t i = 0; i < k; ++i) mask &= mask - 1;
    return __ffs(mask) - 1;
}

// ---------------------------------------------------------------------------------------
// Where the ids of the short pieces live between K2 and K3: DENSE, one word per PIECE (not per byte position: that array was
// written one id per 32-byte sector and read back the same way -- 9x the algorithmic DRAM traffic over the step).
//   by_piece[r]  r = rank of the piece (number of piece starts before it):  the id, when the piece is one token (9 in 10);
//                kPieceMulti | slot, when the merge loop made several tokens of it: they are extras[slot ..], in order;
//                kPieceLong, when the piece is longer than 32 bytes: the long-piece kernels keep its ids in ids_by_pos.
//   extras[]     the tokens of the merged short pieces, allocated a warp at a time (one atomicAdd per 32 pieces).
//   piece_base[t]  pieces before the 2 KiB tile t (K2s counts, tile_scan scans): a piece's rank is its tile's base + a popcount.
// ---------------------------------------------------------------------------------------
constexpr uint32_t kPieceMulti = 0x80000000u;
constexpr uint32_t kPieceLong = 0xFFFFFFFEu;
constexpr uint32_t kPieceTileBytes = kPieceWarps * kPieceRange;      // 2 KiB: one CTA of K2s / K2a
static_assert(kPieceTileBytes == 64 * 32, "K3 derives a word's piece tile as word >> 6");
struct DenseIds {
    uint32_t* by_piece;            // [pieces] <= [total + 1]
    uint32_t* extras;              // [tokens of merged short pieces] <= [total + 1]
    uint32_t extras_cap;
    uint32_t* tile_pieces;         // [n_tiles2k] piece starts per 2 KiB tile
    uint64_t* piece_base;          // [n_tiles2k] exclusive scan of tile_pieces
};

// K2s: one pass over the piece-start flags -- the pieces longer than 32 bytes go to the work list of K2b / K2c (so that the
// long-piece kernels start early, on their own streams), and every 2 KiB tile counts its piece starts.
__global__ void __launch_bounds__(kPieceWarps * 32)
long_scan_kernel(BatchView b, const uint32_t* __restrict__ piece_bits, LongPiece* __restrict__ long_list, uint32_t long_cap,
                 DeviceStatus* status, uint32_t* __restrict__ tile_pieces) {
    const uint32_t lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
    const uint64_t warp = static_cast<uint64_t>(blockIdx.x) * kPieceWarps + wic;
    const uint64_t r0 = warp * kPieceRange;
    const uint64_t r1 = (r0 + kPieceRange < b.total_bytes) ? r0 + kPieceRange : b.total_bytes;
    const bool multi = b.vocab_ids != nullptr;
    // ---- my 16 piece-start bits, and the first piece start after them
    const uint64_t base = r0 + 16ull * lane;
    const uint32_t my = (base < b.total_bytes) ? ((piece_bits[base >> 5] >> (16u * (lane & 1u))) & 0xFFFFu) : 0u;
    uint32_t v = my ? (16u * lane + static_cast<uint32_t>(__ffs(my)) - 1u) : 0xFFFFu;   // offset of my first start in the range
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_down_sync(kFull, v, d); if (lane + d < 32 && o < v) v = o; }
    uint32_t nf_rel = __shfl_down_sync(kFull, v, 1);
    if (lane == 31) nf_rel = 0xFFFFu;
    // a piece that runs past the range ends at the next start beyond it (or at the end of the data)
    const bool any_open = __any_sync(kFull, my != 0 && nf_rel == 0xFFFFu);
    uint64_t beyond = b.total_bytes;
    if (any_open) beyond = next_set_bit(piece_bits, r1, b.total_bytes);
    const uint64_t nf = (nf_rel == 0xFFFFu) ? beyond : r0 + nf_rel;
    // the only piece of my 16 bytes that can be longer than 32 is the LAST one that starts there (the others end inside
    // them).  The counters are bumped once per CTA, not once per piece: with half a million long pieces (CJK text) the
    // kernel was bound by atomics on three addresses (1.0 ms; 0.24 ms on the bench mix).
    __shared__ uint32_t s_n[2], s_at[2], s_pieces;
    __shared__ unsigned long long s_bytes;
    if (threadIdx.x < 2) s_n[threadIdx.x] = 0;
    if (threadIdx.x == 0) { s_bytes = 0; s_pieces = 0; }
    __syncthreads();
    const uint32_t np = __reduce_add_sync(kFull, static_cast<uint32_t>(__popc(my)));
    if (lane == 0 && np) atomicAdd(&s_pieces, np);
    bool is_long = false, big = false;
    uint32_t k = 0, pv = 0;
    uint64_t pos = 0;
    if (my && r0 < b.total_bytes) {
        pos = base + (31u - static_cast<uint32_t>(__clz(my)));
        if (nf - pos > 32) {
            is_long = true;
            big = (nf - pos) > kBigPiece;
            pv = multi ? b.vocab_ids[find_prompt(b.offsets, b.n_prompts, pos)] : 0u;
            k = atomicAdd(&s_n[big ? 1 : 0], 1u);
            atomicAdd(&s_bytes, static_cast<unsigned long long>(nf - pos));
        }
    }
    __syncthreads();
    if (threadIdx.x < 2 && s_n[threadIdx.x]) s_at[threadIdx.x] = atomicAdd(threadIdx.x ? &status->n_big : &status->n_long, s_n[threadIdx.x]);
    if (threadIdx.x == 2 && s_bytes) atomicAdd(&status->long_bytes, s_bytes);
    if (threadIdx.x == 3) tile_pieces[blockIdx.x] = s_pieces;
    __syncthreads();
    if (is_long) {
        const uint32_t idx = s_at[big ? 1 : 0] + k;
        if (idx < long_cap) { LongPiece lp; lp.start = pos; lp.end = nf; lp.vocab = pv; lp.pad = 0; long_list[big ? long_cap - 1 - idx : idx] = lp; }
        else atomicOr(&status->long_overflow, 1u);
    }
}

// ---------------------------------------------------------------------------------------
// K2a + K2m: the short pieces (<= 32 bytes), in two kernels so that both run with full warps.
//   K2a  bpe_lookup_kernel   every piece once: CoreBPE's `if piece in ranks`.  A warp lists the piece starts of its 512
//        bytes in shared memory and its lanes take them round-robin (a lane that owned 16 BYTES had between one and
//        eight pieces to look up); a hit stores the id at the piece's rank (consecutive lanes, consecutive words) and its
//        flag, a miss goes to the CTA's list of its length class, which the CTA appends to the global list with one atomic
//        per class.
//   K2m  bpe_merge_kernel    the misses, one LANE per piece (merge_piece_in_lane), 32 pieces of one length class per
//        warp ticket -- in the fused version the merge loops ran with 4-5 active lanes, because a warp only had the
//        ~15 misses of its own 512 bytes to spread over its lanes (profiles/ncu_lines_bpe_encode_r01n.txt).
// ---------------------------------------------------------------------------------------
constexpr uint32_t kLookupWarps = 4;
static_assert(kLookupWarps == kPieceWarps, "K2a's CTA is the 2 KiB tile K2s counted");
__global__ void __launch_bounds__(kLookupWarps * 32)
bpe_lookup_kernel(BatchView b, VocabSet vs, const uint32_t* __restrict__ piece_bits, DenseIds dn, MissLists ml, DeviceStatus* status) {
    __shared__ uint16_t s_pos[kLookupWarps][kPieceRange + 2];
    __shared__ uint64_t s_miss0[kLookupWarps * kPieceRange / 13 + 8];
    __shared__ uint64_t s_miss1[kLookupWarps * kPieceRange / 7 + 8];
    __shared__ uint64_t s_miss2[kLookupWarps * kPieceRange / 2 + 8];
    __shared__ uint32_t s_cnt[3], s_base[3], s_nw[kLookupWarps];
    const uint32_t lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    const uint64_t warp = static_cast<uint64_t>(blockIdx.x) * kLookupWarps + wic;
    const uint64_t r0 = warp * kPieceRange;
    const uint8_t* __restrict__ text = b.bytes;
    const bool multi = b.vocab_ids != nullptr;
    const bool in_range = r0 < b.total_bytes;
    const uint64_t r1 = (r0 + kPieceRange < b.total_bytes) ? r0 + kPieceRange : b.total_bytes;
    uint32_t n_w = 0;
    if (in_range) {
        // ---- the piece starts of my range, in order, as offsets
        const uint64_t base = r0 + 16ull * lane;
        const uint32_t my = (base < b.total_bytes) ? ((piece_bits[base >> 5] >> (16u * (lane & 1u))) & 0xFFFFu) : 0u;
        const uint32_t cnt = __popc(my);
        uint32_t incl = cnt;
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += o; }
        n_w = __shfl_sync(kFull, incl, 31);
        uint32_t slot = incl - cnt;
        for (uint32_t bits = my; bits; bits &= bits - 1) s_pos[wic][slot++] = static_cast<uint16_t>(16u * lane + static_cast<uint32_t>(__ffs(bits)) - 1u);
    }
    if (lane == 0) s_nw[wic] = n_w;
    __syncthreads();
    if (in_range) {
        // rank of my first piece: the tile's base + the pieces of the warps before me
        uint64_t rank0 = dn.piece_base[blockIdx.x];
        for (uint32_t w = 0; w < wic; ++w) rank0 += s_nw[w];
        // the last piece ends at the next start beyond the range (or at the end of the data)
        uint64_t beyond = b.total_bytes;
        if (n_w) beyond = next_set_bit(piece_bits, r1, b.total_bytes);
        TablesView T = vs.v[0];
        uint32_t vid = 0;
        for (uint32_t i = lane; i < n_w; i += 32) {
            const uint32_t off = s_pos[wic][i];
            const uint64_t pos = r0 + off;
            const uint64_t end = (i + 1 < n_w) ? r0 + s_pos[wic][i + 1] : beyond;
            if (end - pos > 32) { dn.by_piece[rank0 + i] = kPieceLong; continue; }     // long piece: K2b / K2c
            const uint32_t len = static_cast<uint32_t>(end - pos);
            if (multi) {
                const uint32_t pv = b.vocab_ids[find_prompt(b.offsets, b.n_prompts, pos)];
                if (pv != vid) { vid = pv; T = vs.v[vid]; }
            }
            const uint32_t tok = (len == 1) ? T.byte2id[text[pos]] : whole_piece_lookup(T, text + pos, len);   // a byte is a token
            // (leaving the pieces of 13..32 bytes -- hash over the whole piece, byte-wise verify, one or two lanes active here -- to
            //  K2m, where 32 of them fill a warp, took 0.15 ms off this kernel and put 0.35 ms on that one: profiles/ab_variants_r02x.txt)
            if (tok != kNone) {
                dn.by_piece[rank0 + i] = tok;          // (its token flag is its piece flag: flag_count_kernel ORs the piece flags in)
            } else {
                const uint32_t c = len >= 13 ? 0u : (len >= 7 ? 1u : 2u);
                const uint32_t k = atomicAdd(&s_cnt[c], 1u);
                (c == 0 ? s_miss0 : (c == 1 ? s_miss1 : s_miss2))[k] = pos | ((rank0 + i) << 32);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        const uint32_t n = s_cnt[threadIdx.x];
        uint32_t g = n ? atomicAdd(&status->miss_n[threadIdx.x], n) : 0u;
        if (n && g + n > ml.cap[threadIdx.x]) { atomicOr(&status->miss_overflow, 1u); g = 0xFFFFFFFFu; }
        s_base[threadIdx.x] = g;
    }
    __syncthreads();
#pragma unroll
    for (uint32_t c = 0; c < 3; ++c) {
        const uint32_t n = s_cnt[c], g = s_base[c];
        if (g == 0xFFFFFFFFu) continue;
        const uint64_t* src = c == 0 ? s_miss0 : (c == 1 ? s_miss1 : s_miss2);
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) ml.list[c][g + i] = src[i];
    }
}

__global__ void __launch_bounds__(kPieceWarps * 32)
bpe_merge_kernel(BatchView b, VocabSet vs, const uint32_t* __restrict__ piece_bits, DenseIds dn,
                 uint32_t* __restrict__ tok_bits, MissLists ml, DeviceStatus* status) {
    // (one launch per length class with the shared memory sized by the class -- 12 KB instead of 32 KB for the pieces of 2..12
    //  bytes, eight CTAs a SM instead of six -- gained 3 % at full size and cost a launch per sub-batch: not kept)
    __shared__ uint32_t s_id[kPieceWarps][32][32];   // [warp][part][lane]
    __shared__ uint32_t s_rk[kPieceWarps][32][32];
    const uint32_t lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
    const uint8_t* __restrict__ text = b.bytes;
    const bool multi = b.vocab_ids != nullptr;
    uint32_t* sid = &s_id[wic][0][lane];
    uint32_t* srk = &s_rk[wic][0][lane];
    if (status->miss_overflow) return;
    TablesView T = vs.v[0];
    uint32_t vid = 0;
    // (a TMA-staged hot slice of the pair table, probed before the L2-resident table, made this kernel 2x slower:
    //  profiles/ab_variants_r02k.txt, DESIGN.md section 4)
#pragma unroll 1
    for (uint32_t c = 0; c < 3; ++c) {     // longest class first
        const uint32_t n = status->miss_n[c];
        const uint64_t* __restrict__ list = ml.list[c];
        for (;;) {
            uint32_t t0 = 0;
            if (lane == 0) t0 = atomicAdd(&status->miss_next[c], 32u);
            t0 = __shfl_sync(kFull, t0, 0);
            if (t0 >= n) break;
            const uint32_t i = t0 + lane;
            uint32_t alive = 0, rank = 0;
            if (i < n) {
                const uint64_t e = list[i];
                const uint64_t pos = e & 0xFFFFFFFFull;
                rank = static_cast<uint32_t>(e >> 32);
                const uint64_t end = next_set_bit(piece_bits, pos + 1, b.total_bytes);
                if (multi) {
                    const uint32_t pv = b.vocab_ids[find_prompt(b.offsets, b.n_prompts, pos)];
                    if (pv != vid) { vid = pv; T = vs.v[vid]; }
                }
                alive = merge_piece_in_lane(T, text, pos, static_cast<uint32_t>(end - pos), sid, srk, tok_bits);
            }
            // the warp's tokens go to one contiguous stretch of `extras` (one atomic per 32 pieces); the piece's word names its slot
            const uint32_t cnt = __popc(alive);
            uint32_t incl = cnt;
#pragma unroll
            for (uint32_t d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += o; }
            const uint32_t total = __shfl_sync(kFull, incl, 31);
            uint32_t base = 0;
            if (lane == 0 && total) base = atomicAdd(&status->extra_n, total);
            base = __shfl_sync(kFull, base, 0);
            if (cnt) {
                uint32_t slot = base + incl - cnt;
                if (slot + cnt <= dn.extras_cap) {
                    dn.by_piece[rank] = kPieceMulti | slot;
                    for (uint32_t bits = alive; bits; bits &= bits - 1) dn.extras[slot++] = sid[(static_cast<uint32_t>(__ffs(bits)) - 1u) * 32];
                } else atomicOr(&status->miss_overflow, 1u);
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------
// K2b: pieces longer than one window.  One WARP per piece (work list filled by K2, taken with an
// atomic ticket).  The piece's parts live as a compact array in its own slice of per-byte scratch:
//   id[i]  token id of part i            (ids_by_pos slice)
//   rk[i]  rank of the pair (i, i+1), kNone when none / last part
// Phase A, "batched rounds": every occurrence of the current minimum rank r* merges into the SAME
// token, so all non-overlapping occurrences (leftmost first, as the sequential loop would take them)
// are merged in one round -- unless a pair created on the way ranks below r*, which the sequential
// loop would take first: the round is then cut after the leftmost such merge (exact, SURVEY.md H3).
// Runs of one character or of a short period collapse in O(log n) rounds this way.
// Phase B, "list rounds": when a batched round no longer merges a useful fraction, the array turns
// into a linked list; each lane caches the minimum of a contiguous chunk, a round is one warp argmin,
// one merge, two table lookups and a re-scan of the chunks that changed.
// ---------------------------------------------------------------------------------------
struct LongScratch {
    uint32_t* rank;   // u32 per byte position
    uint32_t* aux0;   // phase A: rank of the new left pair  | phase B: next alive part
    uint32_t* aux1;   // phase A: rank of the new right pair | phase B: previous alive part
};

__device__ __forceinline__ uint32_t warp_min_u32(uint32_t v) {
#pragma unroll
    for (uint32_t d = 16; d; d >>= 1) { const uint32_t o = __shfl_xor_sync(kFull, v, d); v = o < v ? o : v; }
    return v;
}

// one 32-element chunk of the selection: which pairs (i, i+1) with rank == rmin merge this round.
// carry = number (parity matters) of consecutive candidates ending just before this chunk.
__device__ __forceinline__ bool select_chunk(uint32_t r, uint32_t rmin, uint32_t lane, uint32_t& carry, uint32_t& sel_ballot) {
    const bool cand = (r == rmin);
    const uint32_t C = __ballot_sync(kFull, cand);
    const uint32_t z = ~C & lanemask_lt(lane);
    const uint32_t s = z ? (32u - __clz(z)) : 0u;             // first lane of the run of candidates ending at me
    const uint32_t cnt = lane - s + (s == 0 ? carry : 0u);    // consecutive candidates right before me
    const bool sel = cand && !(cnt & 1u);
    sel_ballot = __ballot_sync(kFull, sel);
    const uint32_t nz = ~C;
    carry = nz ? static_cast<uint32_t>(__clz(nz)) : (carry + 32u);   // leading ones of C = candidates at the top
    return sel;
}

// One batched round (phase A) by ONE warp on the compact arrays id[] / rk[] of m parts: merges every non-overlapping
// occurrence (leftmost first) of the minimum rank rmin, cut after the leftmost merge that creates a pair ranking below
// rmin (the sequential loop would take that pair next).  a0 / a1 are scratch of m words.  Leaves dead slots (id == kNone)
// for array_compact().
__device__ __forceinline__ void array_round(const TablesView& T, uint32_t* id, uint32_t* rk, uint32_t* a0, uint32_t* a1,
                                            uint32_t m, uint32_t rmin, uint32_t lane) {
    // A1: select, look up the pairs each merge creates, find the cut
    uint32_t carry = 0, prevS = 0, cut = kNone;
    for (uint32_t base = 0; base < m && cut == kNone; base += 32) {
        const uint32_t i = base + lane;
        const uint32_t r = (i + 1 < m) ? rk[i] : kNone;
        uint32_t S;
        const bool sel = select_chunk(r, rmin, lane, carry, S);
        bool viol = false;
        if (sel) {
            const bool selm2 = (lane >= 2) ? ((S >> (lane - 2)) & 1u) : ((prevS >> (30 + lane)) & 1u);
            uint32_t L = kNone, R = kNone;
            if (i > 0) L = pair_lookup(T, selm2 ? rmin : id[i - 1], rmin);
            if (i + 2 < m) R = pair_lookup(T, rmin, id[i + 2]);
            a0[i] = L;
            a1[i] = R;
            viol = (L < rmin) || (R < rmin);
        }
        const uint32_t V = __ballot_sync(kFull, viol);
        if (V) cut = base + (__ffs(V) - 1);
        prevS = S;
    }
    __syncwarp();
    // A2: apply the merges up to the cut, in place (two sub-steps per chunk: right ranks, then left ranks)
    carry = 0; prevS = 0;
    for (uint32_t base = 0; base < m && base <= cut; base += 32) {
        const uint32_t i = base + lane;
        const uint32_t r = (i + 1 < m) ? rk[i] : kNone;
        uint32_t S;
        const bool sel = select_chunk(r, rmin, lane, carry, S);
        const bool app = sel && i <= cut;
        const bool selm2 = (lane >= 2) ? ((S >> (lane - 2)) & 1u) : ((prevS >> (30 + lane)) & 1u);
        uint32_t L = kNone;
        if (app) {
            L = a0[i];
            id[i] = rmin;             // rank == id of the merged token
            id[i + 1] = kNone;        // partner dies
            rk[i] = a1[i];
        }
        __syncwarp();
        if (app && i > 0) rk[selm2 ? i - 2 : i - 1] = L;
        __syncwarp();
        prevS = S;
    }
}
// squeeze the dead slots out (one warp); kPosBits != 0: rk[] holds list-mode keys, turned back into ranks.
// Returns the new part count; rmin_out = the smallest rank left.
template <uint32_t kPosBits>
__device__ __forceinline__ uint32_t array_compact(uint32_t* id, uint32_t* rk, uint32_t m, uint32_t lane, uint32_t& rmin_out) {
    uint32_t out = 0, nmin = kNone;
    for (uint32_t base = 0; base < m; base += 32) {
        const uint32_t i = base + lane;
        const uint32_t myid = (i < m) ? id[i] : kNone;
        uint32_t myrk = (i < m) ? rk[i] : kNone;
        if (kPosBits && myrk != kNone) myrk >>= kPosBits;      // kNoKey == kNone
        const bool keep = myid != kNone;
        const uint32_t K = __ballot_sync(kFull, keep);
        const uint32_t pos = out + __popc(K & lanemask_lt(lane));
        __syncwarp();
        if (keep) { id[pos] = myid; rk[pos] = myrk; nmin = myrk < nmin ? myrk : nmin; }
        out += __popc(K);
    }
    __syncwarp();
    rmin_out = warp_min_u32(nmin);
    return out;
}

constexpr uint32_t kListMax = 65535;
constexpr uint32_t kMedSmem = 256;   // bytes: pieces up to this size keep their merge state in shared memory

// phase B, multi-merge form: up to 32 merges per round, still in the EXACT order of the sequential loop.
// Each lane proposes the minimum pair of its chunk and looks up -- all lanes at once, one table round trip -- the two
// pairs its merge would create.  The proposals are then taken in ascending (rank, position) order while that order is
// provably what the sequential loop would do:
//   * a proposal is only taken while its key is below `bound` = the smallest key of anything that might have to come
//     first: the pairs created by the merges taken so far, and the second-smallest pair of every lane whose proposal
//     has been consumed (its other pairs were not proposed);
//   * a proposal that shares a part with a merge already taken is dropped (what replaced it is covered by `bound`);
//     one that merely neighbours such a merge still exists but its looked-up pairs are stale: the round ends there.
// The global minimum is always taken, so every round makes progress.  A 4 KiB piece of random letters needs ~250 such
// rounds instead of ~2 500 single-merge rounds.
__device__ __forceinline__ bool key_less(uint32_t r1, uint32_t p1, uint32_t r2, uint32_t p2) { return r1 < r2 || (r1 == r2 && p1 < p2); }

__device__ __forceinline__ void list_rounds_multi(const TablesView& T, uint32_t* id, uint32_t* rk, uint32_t* link, uint32_t* nid,
                                                  uint32_t m, uint32_t lane) {
    constexpr uint32_t kNoPrev = 0xFFFFu;
    for (uint32_t i = lane; i < m; i += 32) {
        link[i] = ((i + 1) << 16) | (i ? i - 1 : kNoPrev);
        nid[i] = (i + 1 < m) ? id[i + 1] : kNone;
    }
    __syncwarp();
    const uint32_t c = ((m + 31) / 32) | 1u;      // odd: when the state is in shared memory the lanes' chunks start in 32 different banks
    const uint32_t lo = lane * c < m ? lane * c : m;
    const uint32_t hi = lo + c < m ? lo + c : m;
    for (;;) {
        // -- my chunk's smallest and second-smallest pair, 16 loads in flight
        uint32_t m1 = kNone, p1 = 0, m2 = kNone, p2 = 0;
        for (uint32_t xb = lo; xb < hi; xb += 16) {
            uint32_t v[16];
#pragma unroll
            for (uint32_t t = 0; t < 16; ++t) v[t] = (xb + t < hi) ? rk[xb + t] : kNone;
#pragma unroll
            for (uint32_t t = 0; t < 16; ++t) {
                if (v[t] < m1) { m2 = m1; p2 = p1; m1 = v[t]; p1 = xb + t; }
                else if (v[t] < m2) { m2 = v[t]; p2 = xb + t; }
            }
        }
        if (!__any_sync(kFull, m1 != kNone)) break;
        // -- my proposal (x, its partner j, the parts around them) and the two pairs the merge would create
        const bool valid = m1 != kNone;
        const uint32_t x = p1, r = m1;
        uint32_t j = 0, q = kNoPrev, k = m, L = kNone, R = kNone;
        if (valid) {
            const uint32_t li = link[x];
            j = li >> 16; q = li & 0xFFFFu;
            k = link[j] >> 16;
            const uint32_t idk = nid[j];
            const uint32_t idq = (q != kNoPrev) ? id[q] : 0u;
            pair_lookup2(T, r, idk, k < m, idq, r, q != kNoPrev, R, L);
        }
        // -- take proposals in ascending key order while the sequential loop would.  Lanes own ascending chunks, so
        //    (rank, lane) orders the proposals exactly like (rank, position): one redux names the next one.
        // what my merge, if taken, puts into `bound`: the smaller of its two new pairs and my chunk's second minimum ...
        uint32_t c_r = m2, c_p = p2;
        if (key_less(L, q, c_r, c_p)) { c_r = L; c_p = q; }
        if (key_less(R, x, c_r, c_p)) { c_r = R; c_p = x; }
        const uint32_t xq = x | (q << 16), jk = j | (k << 16);
        bool pending = valid, accepted = false;
        uint32_t bound_r = kNone, bound_p = 0xFFFFFFFFu;
        for (;;) {
            const uint32_t best = __reduce_min_sync(kFull, pending ? ((r << 5) | lane) : kNone);
            if (best == kNone) break;
            const uint32_t s = best & 31u, br = best >> 5;
            const uint32_t sxq = __shfl_sync(kFull, xq, s), sjk = __shfl_sync(kFull, jk, s);
            const uint32_t bp = sxq & 0xFFFFu, sq = sxq >> 16, sj = sjk & 0xFFFFu, sk = sjk >> 16;
            if (!key_less(br, bp, bound_r, bound_p)) break;
            // against every merge already taken this round (u = mine, if I was taken):
            //   gone   the proposal shares a part with u's pair: it no longer exists; what replaced it is in `bound`
            //   stale  it still exists but u changed a neighbour, so its looked-up pairs are out of date: it has to wait
            //          for the next round -- and everything after it in key order with it
            const uint32_t gone_here = (accepted && (j == bp || x == sj)) ? 1u : 0u;
            const uint32_t near_here = (accepted && (x == sq || x == bp || x == sj || x == sk || j == sq || j == bp || j == sj || j == sk ||
                                                     q == bp || q == sj || k == bp || k == sj)) ? 2u : 0u;
            const uint32_t flags = __reduce_or_sync(kFull, gone_here | near_here);
            const bool gone = flags & 1u;
            if (!gone && (flags & 2u)) break;
            if (lane == s) { pending = false; accepted = !gone; }
            // ... or, if it lost a part to an earlier merge, only my chunk's second minimum
            const uint32_t sr = __shfl_sync(kFull, gone ? m2 : c_r, s), sp = __shfl_sync(kFull, gone ? p2 : c_p, s);
            if (key_less(sr, sp, bound_r, bound_p)) { bound_r = sr; bound_p = sp; }
        }
        // -- apply the merges that were taken (their neighbourhoods are disjoint)
        if (accepted) {
            id[x] = r; id[j] = kNone; rk[j] = kNone; rk[x] = R;
            link[x] = (k << 16) | q;
            nid[x] = nid[j];
            if (k < m) link[k] = (link[k] & 0xFFFF0000u) | x;
            if (q != kNoPrev) { rk[q] = L; nid[q] = r; }
        }
        __syncwarp();
    }
}

// phase B, parallel-cut form: every thread of a group of kWarps warps proposes the minimum pair of its chunk of the
// piece, all proposals look up the two pairs their merge would create at once (one table round trip), and ONE min
// reduction decides which of them the sequential loop would have taken next, in order:
//   key(pair) = rank << kPosBits | position          (the sequential loop takes pairs in ascending key order)
//   a proposal S with key a_S is followed, if taken, by nothing smaller than  c_S = min(second-smallest key of S's
//   chunk, keys of the two pairs S creates);  so another proposal L may be taken in the same round only if NOT
//   (a_S < a_L and c_S <= a_L)  for every S, i.e. iff  a_L < cut1 = min_S max(a_S + 1, c_S);
//   two proposals closer than three live parts touch each other's looked-up neighbourhood: the later one (larger key)
//   has to wait, and everything after it: cut2 = min key of those.  Found through a claim array (atomicMin of the key on
//   the two parts of each proposed pair; a proposal that sees a smaller claim on one of its four parts is the later one).
// Taken = key < min(cut1, cut2): their neighbourhoods are disjoint, they apply in parallel.  The global minimum is always
// taken.  With P chunks about 1.2 sqrt(P) merges go through per round on random text (the first chunk hit twice ends the
// prefix): a 4 KiB random word is ~60 rounds of 256 threads instead of ~1 200 single-merge rounds.  tools/model_parcut.py
// checks the rule against the sequential loop on random rank orders.
// On entry id[] / kk[] hold the ids and RANKS of the compact parts; kk[] is converted to keys here.
constexpr uint32_t kNoKey = 0xFFFFFFFFu;
// Returns true when no pair is left.  Pairs of ONE rank are strictly ordered by position, so a stretch of them (a period,
// "xyzxyz...") goes one merge per round here: after three rounds in a row that were cut by a pair of the rank just taken
// the function returns false and the caller does a batched round (array_compact + array_round), which takes them all.
// s_red: 3 * kWarps + 2 words of shared memory (kWarps > 1 only).
// dirty != nullptr (one word per thread): a thread keeps its proposal -- chunk minima, neighbours, the two looked-up pairs --
// from round to round and recomputes only after its merge was taken, after a conflict, or after another thread's merge wrote
// into its chunk (the writer marks the owner).  Per round ~20 of 512 proposals are taken; without this the other ~490 threads
// redid the chunk scan and both table probes every round (160 warp instructions per merge, profiles/ncu_lines_bpe_list_r01n.txt).
template <uint32_t kWarps, uint32_t kPosBits>
__device__ __forceinline__ bool list_rounds_par(const TablesView& T, uint32_t* id, uint32_t* kk, uint32_t* link, uint32_t* claim,
                                                uint32_t m, uint32_t* s_red, uint32_t* dirty = nullptr) {
    constexpr uint32_t kNoPrev = 0xFFFFu, kPosMask = (1u << kPosBits) - 1u, P = kWarps * 32;
    const uint32_t tid = threadIdx.x % P, lane = tid & 31, wid = tid >> 5;
    auto group_sync = [&]() { if (kWarps == 1) __syncwarp(); else __syncthreads(); };
    for (uint32_t i = tid; i < m; i += P) {
        const uint32_t r = kk[i];
        kk[i] = (r == kNone) ? kNoKey : ((r << kPosBits) | i);
        link[i] = ((i + 1) << 16) | (i ? i - 1 : kNoPrev);
        claim[i] = kNoKey;
    }
    if (dirty) dirty[tid] = 0;
    uint32_t* const eq_flag = s_red + 2 * kWarps;     // [2], by round parity
    if (kWarps > 1 && tid == 0) { eq_flag[0] = 0; eq_flag[1] = 0; }
    group_sync();
    uint32_t eq_run = 0;
    uint32_t c = (m + P - 1) / P;
    if (c > 1) c |= 1u;                               // odd: the threads' chunks start in different banks
    const uint32_t lo = tid * c < m ? tid * c : m;
    const uint32_t hi = lo + c < m ? lo + c : m;
    const uint32_t inv_c = (1u << 20) / c + 1u;       // owner of position p = (p * inv_c) >> 20  (exact for p < 4096)
    bool have = false;
    uint32_t m1 = kNoKey, m2 = kNoKey, j = 0, q = kNoPrev, k = m, Lk = kNoKey, Rk = kNoKey;
    for (uint32_t round = 0;; ++round) {
        if (dirty && have && dirty[tid]) have = false;
        if (!have) {
            if (dirty) dirty[tid] = 0;
            // -- smallest and second-smallest key of my chunk
            // (eight loads in flight, two independent min chains: this scan is on the critical path of the round)
            m1 = kNoKey; m2 = kNoKey;
            uint32_t n1 = kNoKey, n2 = kNoKey;
            uint32_t xb = lo;
            for (; xb + 8 <= hi; xb += 8) {            // whole batches: no bounds checks
                uint32_t v[8];
#pragma unroll
                for (uint32_t t = 0; t < 8; ++t) v[t] = kk[xb + t];
#pragma unroll
                for (uint32_t t = 0; t < 8; t += 2) {
                    const uint32_t a = v[t], b = v[t + 1];
                    const uint32_t ha = a > m1 ? a : m1, hb = b > n1 ? b : n1;
                    m2 = ha < m2 ? ha : m2; n2 = hb < n2 ? hb : n2;
                    m1 = a < m1 ? a : m1; n1 = b < n1 ? b : n1;
                }
            }
            if (xb < hi) {                             // the rest: one predicated batch
                uint32_t v[8];
#pragma unroll
                for (uint32_t t = 0; t < 8; ++t) v[t] = (xb + t < hi) ? kk[xb + t] : kNoKey;
#pragma unroll
                for (uint32_t t = 0; t < 8; t += 2) {
                    const uint32_t a = v[t], b = v[t + 1];
                    const uint32_t ha = a > m1 ? a : m1, hb = b > n1 ? b : n1;
                    m2 = ha < m2 ? ha : m2; n2 = hb < n2 ? hb : n2;
                    m1 = a < m1 ? a : m1; n1 = b < n1 ? b : n1;
                }
            }
            {   // merge the two chains: smallest and second smallest of {m1, m2, n1, n2}
                const uint32_t lo1 = m1 < n1 ? m1 : n1, hi1 = m1 < n1 ? n1 : m1;
                const uint32_t s2 = m2 < n2 ? m2 : n2;
                m1 = lo1; m2 = hi1 < s2 ? hi1 : s2;
            }
            // -- my proposal: parts q | x j | k, and the pairs (q, xj) and (xj, k)
            Lk = kNoKey; Rk = kNoKey;
            if (m1 != kNoKey) {
                const uint32_t x = m1 & kPosMask, r = m1 >> kPosBits;
                const uint32_t li = link[x];
                j = li >> 16; q = li & 0xFFFFu;
                k = link[j] >> 16;
                const uint32_t idk = (k < m) ? id[k] : 0u;
                const uint32_t idq = (q != kNoPrev) ? id[q] : 0u;
                uint32_t R, L;
                pair_lookup2(T, r, idk, k < m, idq, r, q != kNoPrev, R, L);
                if (R != kNone) Rk = (R << kPosBits) | x;
                if (L != kNone) Lk = (L << kPosBits) | q;
            }
            have = dirty != nullptr;
        }
        const bool valid = m1 != kNoKey;
        const uint32_t x = m1 & kPosMask, r = m1 >> kPosBits;
        uint32_t v = kNoKey;
        bool viol = false;                             // my merge creates a pair that ranks below it: that pair is next, whatever else is there
        if (valid) {
            uint32_t cc = m2 < Lk ? m2 : Lk;
            cc = cc < Rk ? cc : Rk;
            viol = cc <= m1;
            v = cc > m1 + 1u ? cc : m1 + 1u;
            if (v == kNoKey) v = kNoKey - 1u;          // kNoKey is reserved for "no proposal anywhere"
            atomicMin(&claim[x], m1);
            atomicMin(&claim[j], m1);
        }
        group_sync();
        if (kWarps > 1 && tid == 0) eq_flag[(round + 1u) & 1u] = 0;    // nobody reads or sets the other flag any more
        if (valid) {
            uint32_t lowest = claim[x];
            const uint32_t cj = claim[j];
            lowest = cj < lowest ? cj : lowest;
            if (q != kNoPrev) { const uint32_t cq = claim[q]; lowest = cq < lowest ? cq : lowest; }
            if (k < m) { const uint32_t ck = claim[k]; lowest = ck < lowest ? ck : lowest; }
            if (lowest < m1) { v = m1; have = false; } // someone earlier touches my neighbourhood: the round ends before me
        }
        // -- cut = min over the group
        uint32_t cut = __reduce_min_sync(kFull, v);
        if (kWarps > 1) {
            uint32_t* red = s_red + (round & 1u) * kWarps;
            if (lane == 0) red[wid] = cut;
            __syncthreads();
            cut = red[0];
#pragma unroll
            for (uint32_t w = 1; w < kWarps; ++w) { const uint32_t o = red[w]; cut = o < cut ? o : cut; }
        } else {
            __syncwarp();
        }
        if (cut == kNoKey) return true;
        if (kWarps > 1 && tid == 0) CFBPE_DBG_COUNT(6);
        if (kWarps > 1 && valid && m1 < cut) CFBPE_DBG_COUNT(7);
        // -- a pair of the rank I just took ended the round (and not because my own merge creates a lower pair): same-rank stretch
        bool eq = valid && m1 < cut && !viol && (cut >> kPosBits) == (m1 >> kPosBits);
        if (kWarps == 1) eq = __any_sync(kFull, eq);
        else if (eq) eq_flag[round & 1u] = 1u;
        // -- apply what was taken; withdraw the claims
        if (valid) {
            claim[x] = kNoKey; claim[j] = kNoKey;
            if (m1 < cut) {
                id[x] = r; id[j] = kNone;
                kk[j] = kNoKey; kk[x] = Rk;
                link[x] = (k << 16) | q;
                if (k < m) link[k] = (link[k] & 0xFFFF0000u) | x;
                if (q != kNoPrev) kk[q] = Lk;
                have = false;
                if (dirty) {      // the pairs at j and q may belong to other threads' chunks
                    if (j >= hi) dirty[(j * inv_c) >> 20] = 1u;
                    if (q != kNoPrev && q < lo) dirty[(q * inv_c) >> 20] = 1u;
                }
            }
        }
        group_sync();
        if (kWarps > 1) eq = eq_flag[round & 1u] != 0u;
        eq_run = eq ? eq_run + 1u : 0u;
        if (eq_run >= 3u) {
            // how many pairs of that rank are there?  A batched round costs about as much as 3 (warp) to 20 (CTA) of these
            // rounds: it has to take a fair share of the piece (random text repeats a pair a few times; that is not it)
            const uint32_t er = cut >> kPosBits;
            uint32_t cnt = 0;
            for (uint32_t y = lo; y < hi; ++y) cnt += (kk[y] >> kPosBits) == er ? 1u : 0u;
            cnt = __reduce_add_sync(kFull, cnt);
            if (kWarps > 1) {
                uint32_t* sum = s_red + 2 * kWarps + 2;
                if (lane == 0) sum[wid] = cnt;
                __syncthreads();
                cnt = 0;
#pragma unroll
                for (uint32_t w = 0; w < kWarps; ++w) cnt += sum[w];
                __syncthreads();
            }
            if (cnt >= 8u && cnt * 32u >= m) return false;
            eq_run = 0;
        }
    }
}

// one flag per surviving part of a piece (dead slots hold kNone); order along the piece's slice is token order.
// copy_to != nullptr: the state lives in shared memory, the ids go to the slice as well.
__device__ __forceinline__ void flag_parts(const uint32_t* id, uint32_t* copy_to, uint32_t m, uint64_t start,
                                           uint32_t* __restrict__ tok_bits, DeviceStatus* status, uint32_t lane) {
    for (uint32_t base = 0; base < m; base += 32) {
        const uint32_t i = base + lane;
        const uint32_t v = (i < m) ? id[i] : kNone;
        const bool alive = v != kNone;
        if (alive && copy_to) copy_to[i] = v;
        const uint32_t A = __ballot_sync(kFull, alive);
        if (lane == 0 && A) {
            atomicAdd(&status->long_tokens, static_cast<unsigned long long>(__popc(A)));
            const uint64_t pos = start + base;
            const uint32_t sh = static_cast<uint32_t>(pos & 31);
            atomicOr(&tok_bits[pos >> 5], A << sh);
            if (sh && (A >> (32 - sh))) atomicOr(&tok_bits[(pos >> 5) + 1], A >> (32 - sh));
        }
    }
}

constexpr uint32_t kDeferMaxParts = 4096;   // K2c: parts whose merge state fits 64 KB of shared memory
constexpr uint32_t kListSmemBytes = kDeferMaxParts * 16;
constexpr uint32_t kListMaxRank = (1u << 20) - 1u;   // K2c packs rank << 12 | position into 32 bits
// the big pieces bpe_list_kernel takes (from their bytes); bpe_long_kernel keeps the rest
__device__ __forceinline__ bool list_kernel_takes(const TablesView& T, uint32_t n_bytes) { return n_bytes <= kDeferMaxParts && T.n_ranks < kListMaxRank; }


// One warp per CTA: a warp that is deep in the serial chain of a long piece then holds one warp's worth of registers and
// 6 KB of shared memory, not a whole CTA's, so the tail of this kernel can share the SMs with whatever runs next.
constexpr uint32_t kLongWarps = 4;
#ifndef CFBPE_LONG_MIN_CTAS
#define CFBPE_LONG_MIN_CTAS (32 / kLongWarps)     // launch bound: CTAs per SM the register allocation must allow (A/B: 10, 12)
#endif
__global__ void __launch_bounds__(kLongWarps * 32, CFBPE_LONG_MIN_CTAS)
bpe_long_kernel(BatchView b, VocabSet vs, LongPiece* long_list, DeviceStatus* status,
                uint32_t long_cap, uint32_t* __restrict__ ids_by_pos, LongScratch sc, uint32_t* __restrict__ tok_bits) {
    __shared__ uint32_t s_med[kLongWarps][4][kMedSmem];   // [warp][id | rank | aux0 | aux1] of a piece of <= kMedSmem bytes
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_big = status->n_big;
    const uint32_t n_all = status->long_overflow ? 0u : status->n_long + n_big;
    for (;;) {
        uint32_t item = 0;
        if (lane == 0) item = atomicAdd(&status->long_next, 1u);
        item = __shfl_sync(kFull, item, 0);
        if (item >= n_all) break;
        const uint32_t slot = item < n_big ? long_cap - 1 - item : item - n_big;
        const LongPiece lp = long_list[slot];
        const TablesView T = vs.v[lp.vocab];
        const uint8_t* __restrict__ p = b.bytes + lp.start;
        const uint32_t n = static_cast<uint32_t>(lp.end - lp.start);
#ifndef CFBPE_NO_DEFER
        if (item < n_big && list_kernel_takes(T, n)) continue;       // a big piece: bpe_list_kernel has it, from its bytes, at the same time
#endif
        // state of the piece: shared memory for pieces of <= kMedSmem bytes (most of them), else its slice of scratch
        uint32_t* const gid = ids_by_pos + lp.start;
        const bool in_smem = n <= kMedSmem;
        uint32_t* id = in_smem ? s_med[threadIdx.x >> 5][0] : gid;
        uint32_t* rk = in_smem ? s_med[threadIdx.x >> 5][1] : sc.rank + lp.start;
        uint32_t* a0 = in_smem ? s_med[threadIdx.x >> 5][2] : sc.aux0 + lp.start;
        uint32_t* a1 = in_smem ? s_med[threadIdx.x >> 5][3] : sc.aux1 + lp.start;

        // ---- whole-piece shortcut (CoreBPE: `if piece in ranks`)
        if (n <= T.max_token_len) {
            uint32_t t = kNone;
            if (lane == 0) t = piece_lookup(T, p, n);
            t = __shfl_sync(kFull, t, 0);
            if (t != kNone) {
                if (lane == 0) { gid[0] = t; atomicOr(&tok_bits[lp.start >> 5], 1u << (lp.start & 31)); atomicAdd(&status->long_tokens, 1ull); }
                continue;
            }
        }
        // ---- parts = bytes
        uint32_t m = n;
        uint32_t rmin = kNone;
        for (uint32_t i = lane; i < n; i += 32) {
            const uint32_t c0 = p[i];
            id[i] = T.byte2id[c0];
            const uint32_t r = (i + 1 < n) ? T.bytepair[(c0 << 8) | p[i + 1]] : kNone;
            rk[i] = r;
            rmin = r < rmin ? r : rmin;
        }
        rmin = warp_min_u32(rmin);
        __syncwarp();

        // ---- rounds: batched rounds on the compact array while they merge a useful fraction (runs, periods: O(log n)
        //      rounds), list rounds otherwise; a list phase that meets many pairs of one rank comes back for a batched round
        bool deferred = false;
        while (rmin != kNone) {
            array_round(T, id, rk, a0, a1, m, rmin, lane);
            const uint32_t before = m;
            m = array_compact<0>(id, rk, m, lane, rmin);
            const uint32_t merged = before - m;
            if (rmin == kNone || merged * 8u >= m || m <= 32u || m > kListMax) continue;
            // -- list phase
            if (in_smem) {
                if (list_rounds_par<1, 8>(T, id, rk, a0, a1, m, nullptr)) break;
                if (lane == 0) CFBPE_DBG_COUNT(1);
                m = array_compact<8>(id, rk, m, lane, rmin);
                continue;
            }
            if (lane == 0) CFBPE_DBG_COUNT(5);
            list_rounds_multi(T, id, rk, a0, a1, m, lane);
            __syncwarp();
            break;
        }
        if (deferred) continue;
        __syncwarp();
        flag_parts(id, in_smem ? gid : nullptr, m, lp.start, tok_bits, status, lane);
        __syncwarp();
    }
}

// ---- batched rounds by a whole CTA (the warp forms above, array_round / array_compact, walk the array 32 parts at a time:
//      on a 4 KiB piece that is 128 trips per pass, and it was the 0.45 ms head of the long-piece chain).  Thread t owns the
//      contiguous parts [t * c, t * c + c), c = ceil(m / threads) <= kCtaChunk.
constexpr uint32_t kCtaChunk = 16;        // parts per thread: kListWarps * 32 * kCtaChunk >= kDeferMaxParts

// one batched round on the compact arrays id[] / rk[] of m parts (same result as array_round).
// s_scan: blockDim.x + 2 words; s_sel: kDeferMaxParts / 32 words (which pairs merge this round).
__device__ __forceinline__ void cta_array_round(const TablesView& T, uint32_t* id, uint32_t* rk, uint32_t* a0, uint32_t* a1,
                                                uint32_t m, uint32_t rmin, uint32_t* s_scan, uint32_t* s_sel) {
    const uint32_t P = blockDim.x, t = threadIdx.x;
    const uint32_t c = (m + P - 1) / P;
    const uint32_t lo = t * c < m ? t * c : m, hi = lo + c < m ? lo + c : m;
    // -- candidates of my chunk: are they all candidates, and how many consecutive ones end the chunk
    uint32_t tail = 0, all = 1;
    for (uint32_t i = lo; i < hi; ++i) {
        const bool cand = (i + 1 < m) && rk[i] == rmin;
        if (cand) ++tail; else { tail = 0; all = 0; }
    }
    s_scan[t] = (all << 31) | tail;
    if (t == 0) s_scan[P] = kNone;          // the cut
    for (uint32_t w = t; w < kDeferMaxParts / 32; w += P) s_sel[w] = 0;
    __syncthreads();
    // -- consecutive candidates right before my chunk (walk back over the chunks that are candidates throughout); then select
    //    every second pair of a run of candidates, counted from the run's start (overlapping pairs: leftmost first)
    uint32_t cnt = 0;
    for (uint32_t u = t; u > 0 && lo < m;) {
        const uint32_t e = s_scan[--u];
        cnt += e & 0x7FFFFFFFu;
        if (!(e >> 31)) break;
    }
    uint32_t sel_bits = 0;
    for (uint32_t i = lo; i < hi; ++i) {
        const bool cand = (i + 1 < m) && rk[i] == rmin;
        if (cand && !(cnt & 1u)) { sel_bits |= 1u << (i - lo); atomicOr(&s_sel[i >> 5], 1u << (i & 31)); }
        cnt = cand ? cnt + 1 : 0;
    }
    __syncthreads();
    // -- look up the pairs each merge creates, find the cut
    uint32_t m2_bits = 0;
    for (uint32_t bts = sel_bits; bts; bts &= bts - 1) {
        const uint32_t k = static_cast<uint32_t>(__ffs(bts)) - 1u, i = lo + k;
        const bool selm2 = i >= 2 && ((s_sel[(i - 2) >> 5] >> ((i - 2) & 31)) & 1u);     // the pair two to the left merges too: my left neighbour will be rmin
        uint32_t L = kNone, R = kNone;
        if (i > 0) L = pair_lookup(T, selm2 ? rmin : id[i - 1], rmin);
        if (i + 2 < m) R = pair_lookup(T, rmin, id[i + 2]);
        a0[i] = L; a1[i] = R;
        if (selm2) m2_bits |= 1u << k;
        if (L < rmin || R < rmin) atomicMin(&s_scan[P], i);               // the sequential loop would take that new pair next: cut after this merge
    }
    __syncthreads();
    const uint32_t cut = s_scan[P];
    // -- apply the merges up to the cut: right ranks first, then left ranks (a left write may replace a neighbour's right one)
    for (uint32_t bts = sel_bits; bts; bts &= bts - 1) {
        const uint32_t i = lo + static_cast<uint32_t>(__ffs(bts)) - 1u;
        if (i > cut) break;
        id[i] = rmin; id[i + 1] = kNone; rk[i] = a1[i];
    }
    __syncthreads();
    for (uint32_t bts = sel_bits; bts; bts &= bts - 1) {
        const uint32_t k = static_cast<uint32_t>(__ffs(bts)) - 1u, i = lo + k;
        if (i > cut) break;
        if (i > 0) rk[((m2_bits >> k) & 1u) ? i - 2 : i - 1] = a0[i];
    }
    __syncthreads();
}

// squeeze the dead slots out (whole CTA); kPosBits != 0: rk[] holds list-mode keys, turned back into ranks.  Returns the new part
// count; rmin_out = the smallest rank left.  s_scan: blockDim.x + 2 words.
template <uint32_t kPosBits>
__device__ __forceinline__ uint32_t cta_array_compact(uint32_t* id, uint32_t* rk, uint32_t m, uint32_t& rmin_out, uint32_t* s_scan) {
    const uint32_t P = blockDim.x, t = threadIdx.x, lane = t & 31u, wid = t >> 5;
    const uint32_t c = (m + P - 1) / P;
    const uint32_t lo = t * c < m ? t * c : m, hi = lo + c < m ? lo + c : m;
    uint32_t vid[kCtaChunk], vrk[kCtaChunk];
    uint32_t keep = 0, nmin = kNone;
#pragma unroll
    for (uint32_t k = 0; k < kCtaChunk; ++k) {
        const uint32_t i = lo + k;
        vid[k] = (k < c && i < hi) ? id[i] : kNone;
        uint32_t r = (k < c && i < hi) ? rk[i] : kNone;
        if (kPosBits && r != kNone) r >>= kPosBits;                      // kNoKey == kNone
        vrk[k] = r;
        if (vid[k] != kNone) { ++keep; nmin = r < nmin ? r : nmin; }
    }
    // exclusive scan of the keep counts over the CTA; minimum of the ranks kept
    uint32_t x = keep;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(kFull, x, d); if (lane >= d) x += o; }
    nmin = warp_min_u32(nmin);
    if (lane == 31) s_scan[wid] = x;
    if (lane == 0) s_scan[32 + wid] = nmin;
    __syncthreads();                                                     // (also: everybody has read its chunk)
    uint32_t woff = 0, total = 0, rmin = kNone;
    for (uint32_t w = 0; w < (P >> 5); ++w) { const uint32_t v = s_scan[w]; if (w < wid) woff += v; total += v; const uint32_t r = s_scan[32 + w]; rmin = r < rmin ? r : rmin; }
    uint32_t pos = woff + x - keep;
#pragma unroll
    for (uint32_t k = 0; k < kCtaChunk; ++k) if (vid[k] != kNone) { id[pos] = vid[k]; rk[pos] = vrk[k]; ++pos; }
    __syncthreads();
    rmin_out = rmin;
    return total;
}

// K2c: the big pieces (more than kBigPiece bytes, at most kDeferMaxParts), one CTA of kListWarps warps per piece, FROM THEIR
// BYTES -- batched rounds by the whole CTA while they merge a useful fraction, then parallel-cut rounds (list_rounds_par) -- with
// the whole merge state (id | key | link | claim, 16 bytes per part) in 64 KB of dynamic shared memory.  It does not wait for
// K2b any more (which keeps the pieces of 33..kBigPiece bytes and the rare giants): the long-piece chain was K2b's batched
// rounds on global scratch (0.45 ms, one warp per piece) + this kernel (0.58 ms); now the two kernels run side by side.
// A list round costs one table round trip and a few hundred cycles of shared-memory work and takes ~20 merges.
#ifndef CFBPE_LIST_WARPS
#define CFBPE_LIST_WARPS 8
#endif
constexpr uint32_t kListWarps = CFBPE_LIST_WARPS;
static_assert(kListWarps * 32 * kCtaChunk >= kDeferMaxParts, "a thread's chunk of the batched rounds holds kCtaChunk parts");

__global__ void __launch_bounds__(kListWarps * 32, 3)
bpe_list_kernel(BatchView b, VocabSet vs, const LongPiece* __restrict__ long_list, DeviceStatus* status,
                uint32_t long_cap, uint32_t* __restrict__ ids_by_pos, LongScratch sc, uint32_t* __restrict__ tok_bits) {
    CFBPE_DYN_SMEM(s_dyn);
    __shared__ uint32_t s_red[3 * kListWarps + 2];
    __shared__ uint32_t s_item, s_tok;
    __shared__ uint32_t s_dirty[kListWarps * 32];
    __shared__ uint32_t s_scan[kListWarps * 32 + 64];
    __shared__ uint32_t s_sel[kDeferMaxParts / 32];
    const uint32_t n_big = status->long_overflow ? 0u : status->n_big;
    uint32_t* const id = s_dyn;
    uint32_t* const kk = s_dyn + kDeferMaxParts;
    uint32_t* const link = s_dyn + 2 * kDeferMaxParts;
    uint32_t* const claim = s_dyn + 3 * kDeferMaxParts;
    (void)sc;
    for (;;) {
        if (threadIdx.x == 0) s_item = atomicAdd(&status->defer_next, 1u);
        __syncthreads();
        const uint32_t item = s_item;
        __syncthreads();
        if (item >= n_big) break;
        const LongPiece lp = long_list[long_cap - 1 - item];
        const TablesView T = vs.v[lp.vocab];
        const uint32_t n = static_cast<uint32_t>(lp.end - lp.start);
        if (!list_kernel_takes(T, n)) continue;                          // a giant: K2b's global-memory path
        const uint8_t* __restrict__ p = b.bytes + lp.start;
        uint32_t* const gid = ids_by_pos + lp.start;
        // ---- whole-piece shortcut (CoreBPE: `if piece in ranks`)
        if (n <= T.max_token_len) {
            if (threadIdx.x == 0) s_tok = piece_lookup(T, p, n);
            __syncthreads();
            const uint32_t tok = s_tok;
            __syncthreads();
            if (tok != kNone) {
                if (threadIdx.x == 0) { gid[0] = tok; atomicOr(&tok_bits[lp.start >> 5], 1u << (lp.start & 31)); atomicAdd(&status->long_tokens, 1ull); }
                continue;
            }
        }
        // ---- parts = bytes
        uint32_t m = n, rmin = kNone;
        for (uint32_t i = threadIdx.x; i < n; i += kListWarps * 32) {
            const uint32_t c0 = p[i];
            id[i] = T.byte2id[c0];
            const uint32_t r = (i + 1 < n) ? T.bytepair[(c0 << 8) | p[i + 1]] : kNone;
            kk[i] = r;
            rmin = r < rmin ? r : rmin;
        }
        rmin = warp_min_u32(rmin);
        if ((threadIdx.x & 31) == 0) s_scan[threadIdx.x >> 5] = rmin;
        __syncthreads();
        rmin = kNone;
        for (uint32_t w = 0; w < kListWarps; ++w) { const uint32_t r = s_scan[w]; rmin = r < rmin ? r : rmin; }
        __syncthreads();
        // ---- rounds: batched rounds while they merge a useful fraction (runs, periods: O(log n) rounds), list rounds otherwise; a
        //      list phase that meets many pairs of one rank comes back for a batched round
        bool counted = false;
        while (rmin != kNone) {
            cta_array_round(T, id, kk, link, claim, m, rmin, s_scan, s_sel);
            const uint32_t before = m;
            m = cta_array_compact<0>(id, kk, m, rmin, s_scan);
            if (rmin == kNone || (before - m) * 8u >= m || m <= 32u) continue;
            if (!counted && threadIdx.x == 0) { atomicAdd(&status->defer_n, 1u); atomicAdd(&status->defer_parts, static_cast<unsigned long long>(m)); CFBPE_DBG_COUNT(0); }
            counted = true;
            const bool done = list_rounds_par<kListWarps, 12>(T, id, kk, link, claim, m, s_red, s_dirty);
            __syncthreads();
            if (done) break;
            if (threadIdx.x == 0) CFBPE_DBG_COUNT(2);
            m = cta_array_compact<12>(id, kk, m, rmin, s_scan);        // a stretch of same-rank pairs: back to batched rounds
        }
        __syncthreads();
        if (threadIdx.x < 32) flag_parts(id, gid, m, lp.start, tok_bits, status, threadIdx.x);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------
// K3: flags -> dense output.
//   flag_count:   popcount of each tile of kScanTileWords flag words
//   tile_scan:    exclusive scan of the tile counts (single CTA), total -> status->n_tokens
//   emit_compact: out_ids[rank(pos)] = ids_by_pos[pos]; out_offsets[p] = rank(offsets[p]); counts
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t block_reduce_add_256(uint32_t v, uint32_t* s_tmp) {
#pragma unroll
    for (uint32_t d = 16; d; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    if ((threadIdx.x & 31) == 0) s_tmp[threadIdx.x >> 5] = v;
    __syncthreads();
    uint32_t t = 0;
    for (uint32_t w = 0; w < (blockDim.x + 31) / 32; ++w) t += s_tmp[w];
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(256)
flag_count_kernel(uint32_t* __restrict__ tok_bits, const uint32_t* __restrict__ piece_bits, uint64_t n_words, uint32_t* __restrict__ tile_counts) {
    // Every piece starts with a token: the piece flags are token flags.  The K2 kernels only flag the tokens INSIDE pieces (the
    // merged short ones, the long ones); the piece flags are ORed in here, once, word by word -- K2a used to set them one
    // atomic a piece.  All K2 kernels of the (sub-)batch are done: plain stores.
    __shared__ uint32_t s_tmp[8];
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * kScanTileWords;
    uint32_t c = 0;
    for (uint32_t i = threadIdx.x; i < kScanTileWords; i += blockDim.x) {
        const uint64_t w = base + i;
        if (w < n_words) { const uint32_t t = tok_bits[w], f = t | piece_bits[w]; if (f != t) tok_bits[w] = f; c += __popc(f); }
    }
    const uint32_t t = block_reduce_add_256(c, s_tmp);
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = t;
}

// single CTA; n_tiles arbitrary.  token_base (nullable) = ids produced by the sub-batches before this one (a pipelined host call
// chains them on the device), so tile_base and out_offsets are global ranks.  status (nullable) gets the totals.
// Every WARP scans a contiguous run of tiles, 32 at a time with coalesced loads and a running carry (no barrier inside); two
// passes -- the warps' totals first, then the scan with each warp's offset known -- and two barriers in all, whatever n_tiles is.
// (The first form looped over the tiles 1024 at a time with three barriers a trip: 89 us for the 65 536 two-KiB tiles of a
// 134 MB batch; a thread-per-run form read with a 256-byte stride between lanes and was no faster.)
__global__ void __launch_bounds__(1024)
tile_scan_kernel(const uint32_t* __restrict__ tile_counts, uint32_t n_tiles, uint64_t* __restrict__ tile_base,
                 DeviceStatus* status, const uint64_t* __restrict__ token_base) {
    __shared__ uint64_t s_warp[32];
    const uint64_t base0 = token_base ? *token_base : 0;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    const uint32_t per = ((n_tiles + nwarps - 1) / nwarps + 31u) & ~31u;          // tiles per warp, a multiple of 32
    const uint32_t lo = wid * per < n_tiles ? wid * per : n_tiles;
    const uint32_t hi = lo + per < n_tiles ? lo + per : n_tiles;
    uint64_t sum = 0;
    for (uint32_t i = lo + lane; i < hi; i += 32) sum += tile_counts[i];
#pragma unroll
    for (uint32_t d = 16; d; d >>= 1) sum += __shfl_xor_sync(kFull, sum, d);
    if (lane == 0) s_warp[wid] = sum;
    __syncthreads();
    uint64_t carry = base0, total = 0;
    for (uint32_t w = 0; w < nwarps; ++w) { const uint64_t v = s_warp[w]; if (w < wid) carry += v; total += v; }
    for (uint32_t i0 = lo; i0 < hi; i0 += 32) {
        const uint32_t i = i0 + lane;
        const uint64_t v = i < hi ? tile_counts[i] : 0;
        uint64_t x = v;
#pragma unroll
        for (uint32_t d = 1; d < 32; d <<= 1) { const uint64_t o = __shfl_up_sync(kFull, x, d); if (lane >= d) x += o; }
        if (i < hi) tile_base[i] = carry + x - v;
        carry += __shfl_sync(kFull, x, 31);
    }
    if (threadIdx.x == 0 && status) { status->n_tokens = total; status->tok_end = base0 + total; }
}

// The id of the token whose first byte is bit `bit` of flag word w (emit_compact_kernel, emit_window_kernel).  bits / pb: the
// token and piece flags of the word, prev_*: those of the word before; prank: the rank of the first piece that starts in word w.
__device__ __forceinline__ uint32_t token_id_at(const DenseIds& dn, const uint32_t* __restrict__ ids_by_pos, uint64_t w, uint32_t bit,
                                                uint32_t bits, uint32_t pb, uint32_t prev_bits, uint32_t prev_pb, uint64_t prank) {
    const uint32_t below = pb & ((2u << bit) - 1u);                     // piece starts at or before this token, in my word
    const uint32_t nb = __popc(below);
    const uint32_t v = dn.by_piece[prank + nb - 1];                     // the piece this token belongs to
    uint32_t id;
    if (v == kPieceLong) id = ids_by_pos[(w << 5) + bit];               // a long piece: its kernel left the ids by position
    else if (!(v & kPieceMulti)) id = v;                                // the piece is one token
    else {                                                              // k-th token of a merged piece
        uint32_t k;
        const uint32_t before = bits & ((1u << bit) - 1u);              // tokens before me in my word
        if (nb) { const uint32_t q = 31u - static_cast<uint32_t>(__clz(below)); k = __popc(before >> q); }
        else { const uint32_t q = 31u - static_cast<uint32_t>(__clz(prev_pb)); k = __popc(prev_bits >> q) + __popc(before); }   // (a short piece starts at most one word back)
        id = dn.extras[(v & ~kPieceMulti) + k];
    }
    return id;
}

__global__ void __launch_bounds__(256)
emit_compact_kernel(const uint32_t* __restrict__ tok_bits, const uint32_t* __restrict__ piece_bits, uint64_t n_words,
                    const uint64_t* __restrict__ tile_base, DenseIds dn, const uint32_t* __restrict__ ids_by_pos,
                    uint32_t* __restrict__ out_ids, uint64_t out_cap) {
    // one CTA per tile of kScanTileWords (= blockDim.x) flag words, one word per thread.  A token's rank = prefix popcount of the
    // token flags; its id is found through the rank of the PIECE it belongs to (prefix popcount of the piece flags, per 2 KiB tile)
    __shared__ uint32_t s_warp[8], s_pw[8];
    const uint64_t w = static_cast<uint64_t>(blockIdx.x) * kScanTileWords + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t bits = (w < n_words) ? tok_bits[w] : 0u;
    const uint32_t pb = (w < n_words) ? piece_bits[w] : 0u;
    const uint32_t c = __popc(bits), pc = __popc(pb);
    uint32_t x = c, px = pc;
#pragma unroll
    for (uint32_t d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(kFull, x, d), po = __shfl_up_sync(kFull, px, d);
        if (lane >= d) { x += o; px += po; }
    }
    if (lane == 31) { s_warp[wid] = x; s_pw[wid] = px; }
    // the word before mine (a token's piece may have started there): from my neighbour, or from memory for the first lane
    uint32_t prev_bits = __shfl_up_sync(kFull, bits, 1), prev_pb = __shfl_up_sync(kFull, pb, 1);
    if (lane == 0) { prev_bits = (w > 0 && w <= n_words) ? tok_bits[w - 1] : 0u; prev_pb = (w > 0 && w <= n_words) ? piece_bits[w - 1] : 0u; }
    __syncthreads();
    if (!bits) return;
    uint32_t woff = 0;
    for (uint32_t k = 0; k < wid; ++k) woff += s_warp[k];
    uint64_t r = tile_base[blockIdx.x] + woff + (x - c);
    // pieces that start before my word: the 2 KiB tile (64 words = two warps) has its base from the scan of K2s's counts
    const uint64_t prank = dn.piece_base[w >> 6] + ((wid & 1u) ? s_pw[wid - 1] : 0u) + (px - pc);
    uint32_t rest = bits;
    while (rest) {
        const uint32_t bit = __ffs(rest) - 1;
        rest &= rest - 1;
        const uint32_t id = token_id_at(dn, ids_by_pos, w, bit, bits, pb, prev_bits, prev_pb, prank);
        if (r < out_cap) out_ids[r] = id;
        ++r;
    }
}

// out_offsets[p] = number of flags before byte offsets[p]; counts[p] = difference.  One WARP per prompt boundary: the flags of
// the tile before the position are counted eight words per lane (one thread per prompt walked up to 255 words: 38 us).
__global__ void __launch_bounds__(256)
prompt_offsets_kernel(BatchView b, const uint32_t* __restrict__ tok_bits, const uint64_t* __restrict__ tile_base,
                      uint64_t* __restrict__ out_offsets, uint32_t* __restrict__ out_counts, const DeviceStatus* status) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t i = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (i > b.n_prompts) return;
    auto rank_at = [&](uint64_t pos) -> uint64_t {
        if (pos >= b.total_bytes) return status->tok_end;
        const uint64_t w = pos >> 5;
        const uint64_t w0 = (w / kScanTileWords) * kScanTileWords;
        uint32_t c = 0;
        for (uint64_t k = w0 + lane; k < w; k += 32) c += __popc(tok_bits[k]);
        c = __reduce_add_sync(kFull, c);
        return tile_base[w / kScanTileWords] + c + __popc(tok_bits[w] & ((1u << (pos & 31)) - 1u));
    };
    const uint64_t r = rank_at(b.offsets[i]);
    const uint64_t r1 = (i < b.n_prompts && out_counts) ? rank_at(b.offsets[i + 1]) : r;
    if (lane == 0) {
        out_offsets[i] = r;
        if (i < b.n_prompts && out_counts) out_counts[i] = static_cast<uint32_t>(r1 - r);
    }
}

// ---------------------------------------------------------------------------------------
// Decode (SURVEY.md section 8(f) item 2): ids -> bytes.  tiktoken's decode_bytes: the concatenation of the tokens' bytes.
//   decode_len:    length of every token (0xFFFFFFFF + status->bad_utf8-style flag for an id outside the vocabulary),
//                  and the sum per tile of kDecodeTile tokens
//   tile_scan:     (the kernel of K3) exclusive scan of the tile sums
//   decode_copy:   one CTA per tile: scan of the lengths inside the tile, then every thread copies its token's bytes
//   decode_offsets: byte offset of the first token of every sequence
// ---------------------------------------------------------------------------------------
constexpr uint32_t kDecodeTile = 1024;      // tokens per tile (4 per thread)
struct DecodeView {
    const uint32_t* ids;         // packed ids of all sequences
    const uint64_t* id_offsets;  // [n_seqs + 1]
    const uint8_t* vocab_ids;    // [n_seqs] or nullptr
    uint32_t n_seqs;
    uint64_t n_ids;
};

__global__ void __launch_bounds__(256)
decode_len_kernel(DecodeView d, VocabSet vs, uint32_t* __restrict__ lens, uint32_t* __restrict__ tile_sums, DeviceStatus* status) {
    __shared__ uint32_t s_tmp[8];
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * kDecodeTile;
    uint32_t sum = 0;
    for (uint32_t t = threadIdx.x; t < kDecodeTile; t += blockDim.x) {
        const uint64_t i = base + t;
        if (i >= d.n_ids) break;
        uint32_t vid = 0;
        if (d.vocab_ids) vid = d.vocab_ids[find_prompt(d.id_offsets, d.n_seqs, i)];
        const TablesView& T = vs.v[vid];
        const uint32_t id = d.ids[i];
        uint32_t len = 0;
        if (id < T.n_ranks) len = T.tokoff[id + 1] - T.tokoff[id];
        else atomicOr(&status->bad_utf8, 1u);          // reported as "unknown token id" by the decode entry point
        lens[i] = len;
        sum += len;
    }
    const uint32_t total = block_reduce_add_256(sum, s_tmp);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(256)
decode_copy_kernel(DecodeView d, VocabSet vs, const uint32_t* __restrict__ lens, const uint64_t* __restrict__ tile_base,
                   uint8_t* __restrict__ out, uint64_t out_cap) {
    __shared__ uint32_t s_warp[8];
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * kDecodeTile + 4ull * threadIdx.x;   // my four consecutive tokens
    uint32_t l[4], mine = 0;
#pragma unroll
    for (uint32_t t = 0; t < 4; ++t) { l[t] = (base + t < d.n_ids) ? lens[base + t] : 0u; mine += l[t]; }
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = mine;
#pragma unroll
    for (uint32_t s = 1; s < 32; s <<= 1) { const uint32_t o = __shfl_up_sync(kFull, x, s); if (lane >= s) x += o; }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    uint32_t woff = 0;
    for (uint32_t k = 0; k < wid; ++k) woff += s_warp[k];
    uint64_t o = tile_base[blockIdx.x] + woff + (x - mine);
#pragma unroll
    for (uint32_t t = 0; t < 4; ++t) {
        if (base + t >= d.n_ids || !l[t]) continue;
        uint32_t vid = 0;
        if (d.vocab_ids) vid = d.vocab_ids[find_prompt(d.id_offsets, d.n_seqs, base + t)];
        const TablesView& T = vs.v[vid];
        const uint8_t* src = T.blob + T.tokoff[d.ids[base + t]];
        for (uint32_t k = 0; k < l[t]; ++k) if (o + k < out_cap) out[o + k] = src[k];
        o += l[t];
    }
}

// out_offsets[s] = bytes before the first token of sequence s (out_offsets[n_seqs] = total).  One thread per sequence.
__global__ void __launch_bounds__(256)
decode_offsets_kernel(DecodeView d, const uint32_t* __restrict__ lens, const uint64_t* __restrict__ tile_base,
                      uint64_t* __restrict__ out_offsets, const DeviceStatus* status) {
    const uint64_t sidx = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (sidx > d.n_seqs) return;
    const uint64_t i = d.id_offsets[sidx];
    if (i >= d.n_ids) { out_offsets[sidx] = status->tok_end; return; }     // tile_scan left the total there
    const uint64_t tile = i / kDecodeTile;
    uint64_t r = tile_base[tile];
    for (uint64_t k = tile * kDecodeTile; k < i; ++k) r += lens[k];
    out_offsets[sidx] = r;
}

// the status of a sub-batch, stored straight into pinned host memory: a cudaMemcpyAsync would queue behind the previous
// sub-batch's id download on the same copy engine, and the host would learn too late that the next download can start
__global__ void status_publish_kernel(const DeviceStatus* __restrict__ d, DeviceStatus* h) {
    static_assert(sizeof(DeviceStatus) % 4 == 0 && sizeof(DeviceStatus) <= 256, "one word per thread of a 64-thread block");
    const uint32_t n = sizeof(DeviceStatus) / 4;
    if (threadIdx.x < n) reinterpret_cast<volatile uint32_t*>(h)[threadIdx.x] = reinterpret_cast<const uint32_t*>(d)[threadIdx.x];
    __threadfence_system();
}

}  // namespace cfbpe
#include "pretok_lanes.cuh"     // K1, second form: one lane per 16 bytes (uses split_thread<2> for long runs, load16 for unaligned buffers)
