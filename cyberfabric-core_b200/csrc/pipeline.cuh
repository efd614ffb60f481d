// pipeline.cuh -- the launch sequence of one encode pass (shared by libcfbpe.so and the
// non-GPU SIMT-emulator tests so that both run the same kernels in the same order).
//
// The including translation unit supplies three macros:
//   CFBPE_LAUNCH(kernel, grid, block, stream, ...)   launch
//   CFBPE_LAUNCH_SMEM(kernel, grid, block, smem, stream, ...)   launch with dynamic shared memory
//   CFBPE_ZERO(ptr, bytes, stream)                   asynchronous zero fill
//   CFBPE_MARK(prof, idx, stream, begin)             optional per-kernel event record
//   CFBPE_FORK(main, aux, ev) / CFBPE_JOIN(main, aux, ev)   make aux wait for main / main wait for aux
#pragma once
#include "bpe_kernels.cuh"
#include "window.cuh"

namespace cfbpe {

struct Workspace {
    uint32_t* piece_bits;   // 1 bit per byte: a piece starts here          [n_words + 2]
    uint32_t* tok_bits;     // 1 bit per byte: a token id lives here        [n_words + 2]
    uint32_t* ids_by_pos;   // token id at the byte position of its first byte [total]
    LongScratch lscratch;   // K2b per-byte state                            [total] each
    LongPiece* long_list;
    uint32_t long_cap;
    uint32_t* tile_counts;  // [n_tiles]
    uint64_t* tile_base;    // [n_tiles]
    DeviceStatus* status;
    MissLists miss;         // K2a -> K2m: short pieces that need the merge loop, by length class
    SplitFix* fix_list;     // K1 -> fixup: walkers that stopped in an undecided state (at most one per 16-byte block)   [total / 16 + 2]
    uint32_t fix_cap;
    DenseIds dense;         // ids of the short pieces, one word per piece; extras; piece counts / bases per 2 KiB tile
    uint32_t* pstart_bits;  // 1 bit per byte: a prompt starts here (and one at the end of the data)   [n_words + 2]
    uint32_t* block_prompt; // the prompt that holds the first byte of every 512-byte block           [total / 512 + 2]
};

// the slice of the miss lists that belongs to a sub-batch of `len` bytes starting at byte o0 (k-th sub-batch)
inline MissLists slice_miss(const MissLists& all, uint64_t o0, uint64_t len, uint32_t k) {
    MissLists m;
    for (uint32_t c = 0; c < 3; ++c) {     // (entries are 64-bit: position | rank << 32)
        const uint32_t L = miss_class_min_len(c) < 2 ? 2u : miss_class_min_len(c);   // no one-byte piece is ever a miss
        m.list[c] = all.list[c] + o0 / L + 2ull * k;
        m.cap[c] = static_cast<uint32_t>(len / L + 2);
    }
    return m;
}
inline uint64_t miss_list_words(uint64_t max_bytes, uint32_t c, uint32_t max_chunks) {
    const uint32_t L = miss_class_min_len(c) < 2 ? 2u : miss_class_min_len(c);
    return max_bytes / L + 2ull * max_chunks + 64;
}

// K2b CTAs per SM (long_grid = 4 x SM count).  8 x 128 threads x 64 registers is the whole register file of an SM: the
// short-piece kernels on the other stream then wait for K2b instead of running beside it.
#ifndef CFBPE_LONG_CTAS
#define CFBPE_LONG_CTAS 8
#endif
constexpr uint32_t kLongCtasPerSm = CFBPE_LONG_CTAS;
#ifndef CFBPE_LIST_CTAS
#define CFBPE_LIST_CTAS 3      // (2 -> 3: the kernel alone 0.72 -> 0.57 ms, the step unchanged: profiles/ab_bench_r02z.txt)
#endif
constexpr uint32_t kListCtasPerSm = CFBPE_LIST_CTAS;   // K2c CTAs (64 KB of shared memory each) per SM

enum KernelIdx { K_SPLIT = 0, K_ENCODE = 1, K_LONG = 2, K_COUNT = 3, K_SCAN = 4, K_EMIT = 5, K_LIST = 6, K_LONGSCAN = 7, K_MERGE = 8, K_WINDOW = 9 };

inline uint64_t n_flag_words(uint64_t total_bytes) { return (total_bytes + 31) >> 5; }
inline uint32_t n_scan_tiles(uint64_t total_bytes) {
    return static_cast<uint32_t>((n_flag_words(total_bytes) + kScanTileWords - 1) / kScanTileWords);
}

// The path in stages, so that a caller with more than one stream can overlap the latency-bound long-piece kernel with
// the throughput-bound short-piece kernel (and, in a pipelined host call, with the next sub-batch):
//   split   zero the flags, K1 split, find the long pieces (K2 in scan mode)
//   long    K2b (+ K2c): pieces longer than 32 bytes               } independent of each other:
//   short   K2: whole-piece lookups and in-lane merges (<= 32 B)   } may run on two streams
//   back    flag_count, tile_scan (chained on the previous sub-batch's token total), emit, prompt offsets
template <typename Stream, typename Prof>
inline void enqueue_split(const BatchView& b, const VocabSet& vs, const UcTables& uc, const Workspace& w, Stream stream, Prof* prof,
                          uint32_t split_grid = 0) {
    const uint64_t nw = n_flag_words(b.total_bytes);
    CFBPE_ZERO(w.status, sizeof(DeviceStatus), stream);
    if (!b.total_bytes) return;
    CFBPE_ZERO(w.piece_bits, (nw + 2) * sizeof(uint32_t), stream);
    CFBPE_ZERO(w.tok_bits, (nw + 2) * sizeof(uint32_t), stream);
    CFBPE_MARK(prof, K_SPLIT, stream, true);
#ifdef CFBPE_SPLIT_LEGACY      // A/B build: the first form of K1, one thread per 64-byte chunk
    const uint64_t n_chunks = (b.total_bytes + kSplitChunk - 1) / kSplitChunk;
    CFBPE_LAUNCH(pretok_split_kernel, static_cast<unsigned>((n_chunks + 255) / 256), 256, stream, b, vs, uc, w.piece_bits, w.status, w.fix_list, w.fix_cap);
#else
    CFBPE_ZERO(w.pstart_bits, (nw + 2) * sizeof(uint32_t), stream);
    CFBPE_LAUNCH(prompt_map_kernel, static_cast<unsigned>((static_cast<uint64_t>(b.n_prompts) + 1 + 255) / 256), 256, stream, b, vs, w.pstart_bits, w.block_prompt, w.status);
    {   // K1: persistent CTAs (the product tables are loaded once per CTA); a warp takes tiles of kSplitWarpOwned 16-byte blocks
        const uint64_t n_blocks16 = (b.total_bytes + 15) / 16;
        const uint32_t n_tiles = static_cast<uint32_t>((n_blocks16 + kSplitWarpOwned - 1) / kSplitWarpOwned);
        const uint32_t n_tabs = b.vocab_ids ? kNumPatterns : 1u;
        const uint32_t cap = split_grid ? split_grid : 148u * CFBPE_SPLIT_CTAS;      // resident CTAs: 148 SMs x CTAs per SM (launch bounds)
        const uint32_t n_ctas = (n_tiles + kSplitCta / 32 - 1) / (kSplitCta / 32);
        CFBPE_LAUNCH_SMEM(pretok_split16_kernel, n_ctas < cap ? n_ctas : cap, kSplitCta, n_tabs * kProdTableBytes, stream,
                          b, vs, uc, w.pstart_bits, w.block_prompt, w.piece_bits, w.status, w.fix_list, w.fix_cap, n_tabs, n_tiles);
    }
#endif
    CFBPE_LAUNCH(pretok_fixup_kernel, 296u, 256, stream, b, vs, uc, w.piece_bits, w.status, w.fix_list, w.fix_cap);   // almost always empty
    CFBPE_MARK(prof, K_SPLIT, stream, false);
    const uint64_t n_warps = (b.total_bytes + kPieceRange - 1) / kPieceRange;
    CFBPE_MARK(prof, K_LONGSCAN, stream, true);
    CFBPE_LAUNCH(long_scan_kernel, static_cast<unsigned>((n_warps + kPieceWarps - 1) / kPieceWarps), kPieceWarps * 32, stream,
                 b, w.piece_bits, w.long_list, w.long_cap, w.status, w.dense.tile_pieces);
    CFBPE_MARK(prof, K_LONGSCAN, stream, false);
}

template <typename Stream, typename Prof>
inline void enqueue_short(const BatchView& b, const VocabSet& vs, const Workspace& w, uint32_t long_grid, Stream stream, Prof* prof) {
    if (!b.total_bytes) return;
    const uint64_t n_warps = (b.total_bytes + kPieceRange - 1) / kPieceRange;
    CFBPE_MARK(prof, K_ENCODE, stream, true);
    const uint32_t n_tiles2k = static_cast<uint32_t>((n_warps + kLookupWarps - 1) / kLookupWarps);
    CFBPE_LAUNCH(tile_scan_kernel, 1u, 1024, stream, w.dense.tile_pieces, n_tiles2k, w.dense.piece_base, static_cast<DeviceStatus*>(nullptr),
                 static_cast<const uint64_t*>(nullptr));      // piece ranks: exclusive scan of K2s's per-tile counts
    CFBPE_LAUNCH(bpe_lookup_kernel, n_tiles2k, kLookupWarps * 32, stream, b, vs, w.piece_bits, w.dense, w.miss, w.status);
    CFBPE_MARK(prof, K_ENCODE, stream, false);
    CFBPE_MARK(prof, K_MERGE, stream, true);
    CFBPE_LAUNCH(bpe_merge_kernel, long_grid + long_grid / 2, kPieceWarps * 32, stream,      // 6 CTAs of 32 KB per SM
                 b, vs, w.piece_bits, w.dense, w.tok_bits, w.miss, w.status);
    CFBPE_MARK(prof, K_MERGE, stream, false);
}

// K2b: the pieces of 33 .. kBigPiece bytes (and the rare giants the list kernel cannot hold), one warp each
template <typename Stream, typename Prof>
inline void enqueue_long(const BatchView& b, const VocabSet& vs, const Workspace& w, uint32_t long_grid, Stream stream, Prof* prof) {
    if (!b.total_bytes) return;
    CFBPE_MARK(prof, K_LONG, stream, true);
    CFBPE_LAUNCH(bpe_long_kernel, (long_grid / 4) * kLongCtasPerSm, kLongWarps * 32, stream, b, vs, w.long_list, w.status, w.long_cap, w.ids_by_pos, w.lscratch, w.tok_bits);
    CFBPE_MARK(prof, K_LONG, stream, false);
}
// K2c: the big pieces, one CTA each, from their bytes -- independent of K2b (its own stream where the caller has one): two 64 KB
// CTAs per SM (long_grid = 4 x SM count), so that the short-piece kernels on the other stream keep ~100 KB of shared memory per SM
template <typename Stream, typename Prof>
inline void enqueue_list(const BatchView& b, const VocabSet& vs, const Workspace& w, uint32_t long_grid, Stream stream, Prof* prof) {
    if (!b.total_bytes) return;
#ifndef CFBPE_NO_DEFER
    CFBPE_MARK(prof, K_LIST, stream, true);
    CFBPE_LAUNCH_SMEM(bpe_list_kernel, (long_grid / 4) * kListCtasPerSm, kListWarps * 32, kListSmemBytes, stream, b, vs, w.long_list, w.status, w.long_cap, w.ids_by_pos, w.lscratch, w.tok_bits);
    CFBPE_MARK(prof, K_LIST, stream, false);
#endif
}

// back = count | scan | emit.  Only the scan reads what the previous sub-batch of a pipelined call produced (token_base), so
// a caller that chains sub-batches waits between count and scan and can let the emits of consecutive sub-batches overlap.
template <typename Stream, typename Prof>
inline void enqueue_count(const BatchView& b, const Workspace& w, Stream stream, Prof* prof) {
    if (!b.total_bytes) return;
    CFBPE_MARK(prof, K_COUNT, stream, true);
    CFBPE_LAUNCH(flag_count_kernel, n_scan_tiles(b.total_bytes), 256, stream, w.tok_bits, w.piece_bits, n_flag_words(b.total_bytes), w.tile_counts);
    CFBPE_MARK(prof, K_COUNT, stream, false);
}
template <typename Stream, typename Prof>
inline void enqueue_scan(const BatchView& b, const Workspace& w, Stream stream, Prof* prof, const uint64_t* token_base) {
    if (b.total_bytes) {
        CFBPE_MARK(prof, K_SCAN, stream, true);
        CFBPE_LAUNCH(tile_scan_kernel, 1u, 1024, stream, w.tile_counts, n_scan_tiles(b.total_bytes), w.tile_base, w.status, token_base);
        CFBPE_MARK(prof, K_SCAN, stream, false);
    } else {
        CFBPE_LAUNCH(tile_scan_kernel, 1u, 32, stream, w.tile_counts, 0u, w.tile_base, w.status, token_base);   // tok_end = base
    }
}
template <typename Stream, typename Prof>
inline void enqueue_emit(const BatchView& b, const Workspace& w, uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets,
                         uint32_t* out_counts, Stream stream, Prof* prof) {
    CFBPE_MARK(prof, K_EMIT, stream, true);
    if (b.total_bytes && out_ids) {
        CFBPE_LAUNCH(emit_compact_kernel, n_scan_tiles(b.total_bytes), 256, stream, w.tok_bits, w.piece_bits, n_flag_words(b.total_bytes), w.tile_base,
                     w.dense, w.ids_by_pos, out_ids, out_cap);
    }
    CFBPE_LAUNCH(prompt_offsets_kernel, static_cast<unsigned>((static_cast<uint64_t>(b.n_prompts) + 1 + 7) / 8), 256, stream,      // a warp per prompt boundary
                 b, w.tok_bits, w.tile_base, out_offsets, out_counts, w.status);
    CFBPE_MARK(prof, K_EMIT, stream, false);
}
template <typename Stream, typename Prof>
inline void enqueue_back(const BatchView& b, const Workspace& w, uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets,
                         uint32_t* out_counts, Stream stream, Prof* prof, const uint64_t* token_base) {
    enqueue_count(b, w, stream, prof);
    enqueue_scan(b, w, stream, prof, token_base);
    enqueue_emit(b, w, out_ids, out_cap, out_offsets, out_counts, stream, prof);
}

// window (truncated encode, after enqueue_emit has written the token offsets and counts of the (sub-)batch): tok_off[p] = rank of
// prompt p's first token, counts[p] = its token count (prompt_offsets_kernel's outputs).  Rows are emitted only when win.rows is set.
template <typename Stream, typename Prof>
inline void enqueue_window(const BatchView& b, const VocabSet& vs, const Workspace& w, const uint64_t* tok_off, const uint32_t* counts,
                           const WindowView& win, Stream stream, Prof* prof) {
    if (!b.n_prompts) return;
    CFBPE_MARK(prof, K_WINDOW, stream, true);
    CFBPE_LAUNCH(window_select_kernel, static_cast<unsigned>((static_cast<uint64_t>(b.n_prompts) + 7) / 8), 256, stream,    // a warp per prompt
                 b, vs, w.tok_bits, w.piece_bits, w.ids_by_pos, counts, win);
    if (b.total_bytes && win.rows) {
        CFBPE_LAUNCH(emit_window_kernel, n_scan_tiles(b.total_bytes), 256, stream, w.tok_bits, w.piece_bits, n_flag_words(b.total_bytes),
                     w.tile_base, w.dense, w.ids_by_pos, b, w.block_prompt, tok_off, counts, win);
    }
    CFBPE_MARK(prof, K_WINDOW, stream, false);
}

// The whole path.  `aux` / `aux2` are streams of their own for the two long-piece kernels (pass the main stream to run everything
// in order); CFBPE_FORK / CFBPE_JOIN order them.  out_ids may be nullptr (count only).  Everything is asynchronous.
template <typename Stream, typename Prof, typename Ev>
inline void enqueue_encode(const BatchView& b, const VocabSet& vs, const UcTables& uc, const Workspace& w,
                           uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets, uint32_t* out_counts,
                           uint32_t long_grid, Stream stream, Stream aux, Stream aux2, Ev ev_fork, Ev ev_join, Ev ev_join2, Prof* prof,
                           const uint64_t* token_base = nullptr) {
    enqueue_split(b, vs, uc, w, stream, prof);
    CFBPE_FORK(stream, aux2, ev_fork);
    enqueue_list(b, vs, w, long_grid, aux2, prof);
    CFBPE_FORK(stream, aux, ev_fork);
    enqueue_long(b, vs, w, long_grid, aux, prof);
    enqueue_short(b, vs, w, long_grid, stream, prof);
    CFBPE_JOIN(stream, aux, ev_join);
    CFBPE_JOIN(stream, aux2, ev_join2);
    enqueue_back(b, w, out_ids, out_cap, out_offsets, out_counts, stream, prof, token_base);
}

}  // namespace cfbpe
