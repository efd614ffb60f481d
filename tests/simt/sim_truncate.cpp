// sim_truncate.cpp -- the truncated encode (csrc/window.cuh after K1..K3) on the CPU SIMT emulator.
// TEST INFRASTRUCTURE: built by tests/simt/simtrunc.py into tests/simt/_build/libcfbpe_sim_truncate.so, loaded only by the
// non-GPU tests of tests/test_truncate.py.  It is the harness of sim_harness.cpp (vocabularies, tables, the other entry points)
// plus one entry point; the kernels are the product sources, compiled unchanged.
#include "sim_harness.cpp"

extern "C" {

// K1..K3 in count mode on host memory, then the window stage: budgets, rows and cut may be NULL; n_long_out (may be NULL) gets
// the number of pieces the long-piece kernels took
__attribute__((visibility("default"))) int sim_encode_truncated(void* const* vocabs, uint32_t n_vocabs, uint32_t n_prompts,
                                                                const uint8_t* bytes, const uint64_t* offsets, const uint8_t* vocab_ids,
                                                                uint32_t max_tokens, uint32_t keep, uint32_t pad_id, const uint32_t* budgets,
                                                                uint32_t* rows, uint32_t* kept, uint32_t* counts, uint64_t* cut,
                                                                uint64_t* n_long_out) {
    const uint64_t total = offsets[n_prompts];
    std::vector<uint8_t> padded(bytes, bytes + total); padded.resize(total + 64);
    BatchView b{padded.data(), offsets, vocab_ids, n_prompts, total};
    VocabSet vs{};
    for (uint32_t i = 0; i < n_vocabs && i < kMaxVocabs; ++i) {
        SimVocab* v = static_cast<SimVocab*>(vocabs[i]);
        vs.v[i] = make_view(v->blob.data(), v->hdr);
    }
    vs.loaded_mask = n_vocabs >= 32 ? 0xFFFFFFFFu : ((1u << n_vocabs) - 1u);
    // the workspace of one sub-batch, as sim_encode_batch lays it out
    const uint64_t nw = n_flag_words(total);
    const uint32_t nt = n_scan_tiles(total);
    std::vector<uint32_t> piece_bits(nw + 2), tok_bits(nw + 2), ids(total + 1, 0xDEADBEEF), rk(total + 1), nx(total + 1), pv(total + 1);
    std::vector<uint32_t> tile_counts(nt + 1);
    std::vector<uint64_t> tile_base(nt + 1);
    std::vector<LongPiece> ll(total / 32 + 1);
    DeviceStatus st{};
    std::vector<SplitFix> fix(total / 16 + 2);
    std::vector<uint64_t> miss[3];
    MissLists ml;
    for (uint32_t c = 0; c < 3; ++c) {
        miss[c].resize(miss_list_words(total, c, 1));
        ml.list[c] = miss[c].data();
        ml.cap[c] = static_cast<uint32_t>(miss[c].size());
    }
    std::vector<uint32_t> pstart(nw + 2), bprompt((total >> kPromptBlockShift) + 2);
    std::vector<uint32_t> by_piece(total + 1, 0xDEADBEEF), extras(total + 1, 0xDEADBEEF), tile_pieces((total >> 11) + 2);
    std::vector<uint64_t> piece_base((total >> 11) + 2);
    Workspace w{piece_bits.data(), tok_bits.data(), ids.data(), LongScratch{rk.data(), nx.data(), pv.data()},
                ll.data(), static_cast<uint32_t>(ll.size()), tile_counts.data(), tile_base.data(), &st, ml, fix.data(), static_cast<uint32_t>(fix.size()),
                DenseIds{by_piece.data(), extras.data(), static_cast<uint32_t>(extras.size()), tile_pieces.data(), piece_base.data()},
                pstart.data(), bprompt.data()};
    // the token offsets and counts the window reads (the library keeps them in the lane's offset and count buffers)
    std::vector<uint64_t> tok_off(static_cast<size_t>(n_prompts) + 1);
    std::vector<uint32_t> tok_counts(static_cast<size_t>(n_prompts) + 1);
    const WindowView win{max_tokens, keep, pad_id, budgets, rows, kept, counts, cut};
    int* prof = nullptr;
    enqueue_encode(b, vs, uc_tables(), w, nullptr, 0, tok_off.data(), tok_counts.data(), 4u, 0, 0, 0, 0, 0, 0, prof);
    enqueue_window(b, vs, w, tok_off.data(), tok_counts.data(), win, 0, prof);
    if (n_long_out) *n_long_out = static_cast<uint64_t>(st.n_long) + st.n_big;
    if (st.bad_utf8) return CFBPE_EILSEQ;
    if (st.long_overflow || st.miss_overflow) return CFBPE_EIO;
    return 0;
}

}  // extern "C"
