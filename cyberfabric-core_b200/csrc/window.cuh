// window.cuh -- truncated encode (cfbpe_encode_truncated): the token window of every prompt, after K3.
//
// For prompt p with c_p tokens, a row length L and an optional budget, the prompt keeps k_p = min(c_p, budget_p, L) tokens:
// its first k_p (HEAD) or its last k_p (TAIL).  Everything the window needs is on the device once prompt_offsets_kernel has
// run: tok_bits flags every token, tile_base + tok_off give every token its rank and every prompt its first rank.  A token flag is
// the token's first byte, except inside a long piece (> 32 bytes): K2b / K2c flag its tokens in order at the piece's first slots
// (and leave their ids at those positions in ids_by_pos), so a cut inside such a piece is the piece start plus the byte lengths of
// the piece's tokens before it.
//   window_select  a warp per prompt: k_p, the default cut, the padding of row p; for a truncated prompt, the byte position of the
//                  token at the cut (a walk over tok_bits from the nearer end of the prompt)
//   emit_window    one thread per flag word, as emit_compact: every token inside its prompt's window goes to rows[p * L + j - lo_p]
// tok_off / counts / rows / kept / cut are indexed by the prompt inside the (sub-)batch; tok_off and tile_base come from the same
// rank chain (global, or shard-local on a multi-device shard), so the in-prompt index of a token is rank - tok_off[p] either way.
#pragma once
#include "bpe_kernels.cuh"

namespace cfbpe {

constexpr uint32_t kKeepHead = 0, kKeepTail = 1;      // CFBPE_KEEP_HEAD / CFBPE_KEEP_TAIL

struct WindowView {
    uint32_t max_tokens;       // L: ids per row
    uint32_t keep;             // kKeepHead | kKeepTail
    uint32_t pad_id;
    const uint32_t* budgets;   // [n] or nullptr (L for every prompt)
    uint32_t* rows;            // [n * L] or nullptr (no ids: emit_window is not launched)
    uint32_t* kept;            // [n] k_p
    uint32_t* counts_out;      // [n] or nullptr: c_p copied here (the device entry; the host paths download the scratch counts)
    uint64_t* cut;             // [n] or nullptr: byte offset of the cut inside the prompt
};

// the (r+1)-th set bit of v from the bottom (from_top = false) or from the top; v holds more than r set bits
__device__ __forceinline__ uint32_t nth_set_bit(uint32_t v, uint32_t r, bool from_top) {
    if (from_top) {
        for (uint32_t i = 0; i < r; ++i) v &= ~(0x80000000u >> __clz(v));
        return 31u - static_cast<uint32_t>(__clz(v));
    }
    for (uint32_t i = 0; i < r; ++i) v &= v - 1u;
    return static_cast<uint32_t>(__ffs(v)) - 1u;
}

// the byte position of the token flagged at q (a flag of prompt [s, e)), by the whole warp: q itself unless q lies in a long piece
__device__ __forceinline__ uint64_t flag_to_byte(const BatchView& b, const VocabSet& vs, const uint32_t* __restrict__ tok_bits,
                                                 const uint32_t* __restrict__ piece_bits, const uint32_t* __restrict__ ids_by_pos,
                                                 uint64_t p, uint64_t s, uint64_t e, uint64_t q, uint32_t lane) {
    // the piece holding q starts at the last piece flag at or before q (the prompt's first byte starts one): 32 words a step back
    uint64_t ps = s;
    for (uint64_t d0 = 0; d0 <= (q >> 5) - (s >> 5); d0 += 32) {
        const uint64_t d = d0 + lane, wp = (q >> 5) - d;
        uint32_t v = 0u;
        if (d <= (q >> 5) - (s >> 5)) { v = piece_bits[wp]; if (d == 0) v &= (2u << (q & 31)) - 1u; if (wp == (s >> 5)) v &= ~0u << (s & 31); }
        const uint32_t h = __ballot_sync(kFull, v != 0u);
        if (h) {
            const uint32_t src = static_cast<uint32_t>(__ffs(h)) - 1u;
            ps = (__shfl_sync(kFull, wp, src) << 5) + 31u - static_cast<uint32_t>(__clz(__shfl_sync(kFull, v, src)));
            break;
        }
    }
    // long: no piece starts in (ps, ps + 32] and the prompt goes on past it (the piece ends at the next start or the prompt's end)
    bool is_long = e > ps + 32;
    if (is_long) {
        const uint64_t a = ps + 1, z = ps + 32;                // the two flag words that hold (ps, ps + 32]
        uint32_t lo = piece_bits[a >> 5] & (~0u << (a & 31));
        if ((z >> 5) == (a >> 5)) lo &= (2u << (z & 31)) - 1u;
        else if (piece_bits[z >> 5] & ((2u << (z & 31)) - 1u)) is_long = false;
        if (lo) is_long = false;
    }
    if (!is_long) return q;
    const TablesView& T = vs.v[b.vocab_ids ? b.vocab_ids[p] : 0u];
    uint32_t sum = 0;                                          // bytes of the piece's tokens flagged in [ps, q)
    for (uint64_t w = (ps >> 5) + lane; w <= (q >> 5); w += 32) {
        uint32_t f = tok_bits[w];
        if (w == (ps >> 5)) f &= ~0u << (ps & 31);
        if (w == (q >> 5)) f &= (1u << (q & 31)) - 1u;
        while (f) {
            const uint32_t bit = static_cast<uint32_t>(__ffs(f)) - 1u;
            f &= f - 1u;
            const uint32_t id = ids_by_pos[(w << 5) + bit];
            sum += T.tokoff[id + 1] - T.tokoff[id];
        }
    }
    return ps + __reduce_add_sync(kFull, sum);
}

// One warp per prompt.  The walk (truncated prompts only, 0 < t < c_p): in-prompt token t has the (t+1)-th token flag of the
// prompt's bytes.  The warp reads 32 flag words a step from the nearer end of the prompt, counts them (popcount + warp scan) and
// the ballot names the word that holds it; flag_to_byte turns the flag into the token's first byte.
__global__ void __launch_bounds__(256)
window_select_kernel(BatchView b, VocabSet vs, const uint32_t* __restrict__ tok_bits, const uint32_t* __restrict__ piece_bits,
                     const uint32_t* __restrict__ ids_by_pos, const uint32_t* __restrict__ counts, WindowView win) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t p = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (p >= b.n_prompts) return;
    const uint32_t c = counts[p];
    uint32_t k = c < win.max_tokens ? c : win.max_tokens;
    if (win.budgets && win.budgets[p] < k) k = win.budgets[p];
    if (lane == 0) { win.kept[p] = k; if (win.counts_out) win.counts_out[p] = c; }
    if (win.rows) {
        uint32_t* row = win.rows + p * win.max_tokens;
        for (uint32_t j = k + lane; j < win.max_tokens; j += 32) row[j] = win.pad_id;
    }
    if (!win.cut) return;
    const uint64_t s = b.offsets[p], e = b.offsets[p + 1];
    const uint32_t t = win.keep == kKeepHead ? k : c - k;      // the in-prompt index of the token at the cut
    if (k == c || t == 0 || t >= c) {       // no walk: nothing dropped, or the cut is at one end of the prompt
        uint64_t at = (t == 0) ? 0 : e - s;                    // (the first token starts at the prompt's first byte)
        if (k == c) at = win.keep == kKeepHead ? e - s : 0;
        if (lane == 0) win.cut[p] = at;
        return;
    }
    const uint64_t w0 = s >> 5, w1 = (e - 1) >> 5;              // the prompt's flag words (inclusive)
    const uint32_t m0 = ~0u << (s & 31), m1 = (e & 31) ? ((1u << (e & 31)) - 1u) : ~0u;
    const bool from_top = c - t < t;
    uint32_t need = from_top ? c - 1u - t : t;                 // flags to pass over before the one we want
    for (uint64_t step = 0;; step += 32) {
        const uint64_t d = step + lane;                        // distance from the end the walk starts at
        const bool in = d <= w1 - w0;
        const uint64_t w = from_top ? w1 - d : w0 + d;
        uint32_t v = 0u;
        if (in) { v = tok_bits[w]; if (w == w0) v &= m0; if (w == w1) v &= m1; }
        const uint32_t n = __popc(v);
        uint32_t x = n;
#pragma unroll
        for (uint32_t sh = 1; sh < 32; sh <<= 1) { const uint32_t o = __shfl_up_sync(kFull, x, sh); if (lane >= sh) x += o; }
        const uint32_t hit = __ballot_sync(kFull, x > need);
        if (hit) {
            const uint32_t src = static_cast<uint32_t>(__ffs(hit)) - 1u;
            const uint64_t q = (__shfl_sync(kFull, w, src) << 5) +
                               nth_set_bit(__shfl_sync(kFull, v, src), need - (__shfl_sync(kFull, x, src) - __shfl_sync(kFull, n, src)), from_top);
            const uint64_t at = flag_to_byte(b, vs, tok_bits, piece_bits, ids_by_pos, p, s, e, q, lane);
            if (lane == 0) win.cut[p] = at - s;
            return;
        }
        need -= __shfl_sync(kFull, x, 31);
    }
}

// One CTA per tile of kScanTileWords flag words, one word per thread: ranks and ids exactly as emit_compact_kernel finds them.
// A token's prompt comes from block_prompt (the prompt holding the first byte of its 512-byte block) and the offsets, moving
// forward through the word -- empty prompts set no prompt-start bit, so the prompt index is not a count of pstart_bits.
// (The word setup repeats emit_compact_kernel's: moving it into a shared inline function changed that kernel's machine code.)
__global__ void __launch_bounds__(256)
emit_window_kernel(const uint32_t* __restrict__ tok_bits, const uint32_t* __restrict__ piece_bits, uint64_t n_words,
                   const uint64_t* __restrict__ tile_base, DenseIds dn, const uint32_t* __restrict__ ids_by_pos, BatchView b,
                   const uint32_t* __restrict__ block_prompt, const uint64_t* __restrict__ tok_off, const uint32_t* __restrict__ counts,
                   WindowView win) {
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
    uint32_t prev_bits = __shfl_up_sync(kFull, bits, 1), prev_pb = __shfl_up_sync(kFull, pb, 1);
    if (lane == 0) { prev_bits = (w > 0 && w <= n_words) ? tok_bits[w - 1] : 0u; prev_pb = (w > 0 && w <= n_words) ? piece_bits[w - 1] : 0u; }
    __syncthreads();
    if (!bits) return;
    uint32_t woff = 0;
    for (uint32_t k = 0; k < wid; ++k) woff += s_warp[k];
    uint64_t r = tile_base[blockIdx.x] + woff + (x - c);
    const uint64_t prank = dn.piece_base[w >> 6] + ((wid & 1u) ? s_pw[wid - 1] : 0u) + (px - pc);
    uint32_t p = block_prompt[(w << 5) >> kPromptBlockShift], cur = ~0u, kp = 0;
    uint64_t lo = 0;                                           // the window of prompt p: ranks [lo, lo + kp)
    uint32_t rest = bits;
    while (rest) {
        const uint32_t bit = __ffs(rest) - 1;
        rest &= rest - 1;
        const uint64_t pos = (w << 5) + bit;
        while (b.offsets[p + 1] <= pos) ++p;                   // (as prompt_at; the 32 bytes of a word lie in one 512-byte block)
        if (p != cur) {
            cur = p;
            kp = win.kept[p];
            lo = tok_off[p] + (win.keep == kKeepHead ? 0 : counts[p] - kp);
        }
        const uint64_t j = r - lo;                             // (wraps for tokens before the window)
        if (j < kp) win.rows[static_cast<uint64_t>(p) * win.max_tokens + j] = token_id_at(dn, ids_by_pos, w, bit, bits, pb, prev_bits, prev_pb, prank);
        ++r;
    }
}

}  // namespace cfbpe
