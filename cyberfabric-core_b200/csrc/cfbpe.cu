// cfbpe.cu -- libcfbpe.so: device context, vocab upload and the C ABI of include/cfbpe.h.
//
// Built for sm_100a only.  There is no CPU path in this library: every entry point that
// computes runs the kernels of bpe_kernels.cuh on the device or returns an error.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/cfbpe.h"

struct ProfEvents;
#define CFBPE_LAUNCH(kernel, grid, block, stream, ...) kernel<<<(grid), (block), 0, (stream)>>>(__VA_ARGS__)
#define CFBPE_LAUNCH_SMEM(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define CFBPE_ZERO(ptr, bytes, stream) cudaMemsetAsync((ptr), 0, (bytes), (stream))
#define CFBPE_MARK(prof, idx, stream, begin) prof_mark((prof), (idx), (stream), (begin))
static inline void prof_mark(ProfEvents* p, int idx, cudaStream_t s, bool begin);
// make `aux` wait for what is queued on `main` so far / make `main` wait for `aux`; no-ops when both are the same stream
#define CFBPE_FORK(main, aux, ev) do { if ((main) != (aux)) { cudaEventRecord((ev), (main)); cudaStreamWaitEvent((aux), (ev), 0); } } while (0)
#define CFBPE_JOIN(main, aux, ev) do { if ((main) != (aux)) { cudaEventRecord((ev), (aux)); cudaStreamWaitEvent((main), (ev), 0); } } while (0)

#include "pipeline.cuh"
#include "pretok_ctx.h"
#include "subbatch.h"
#include "unicode_tables.h"
#include "vocab.h"

using namespace cfbpe;

struct ProfEvents {
    cudaEvent_t ev[CFBPE_NUM_KERNELS][2];
    cudaEvent_t h2d[2], d2h[2], total[2];
    bool launched[CFBPE_NUM_KERNELS];
    uint32_t window_launches;            // K_WINDOW: window_select, + emit_window when rows are wanted
};
static inline void prof_mark(ProfEvents* p, int idx, cudaStream_t s, bool begin) {
    if (!p) return;
    cudaEventRecord(p->ev[idx][begin ? 0 : 1], s);
    p->launched[idx] = true;
}

#include <dlfcn.h>

#include <atomic>
#include <memory>
#include <shared_mutex>
#include <thread>

constexpr int kMaxPipeChunks = 64;
constexpr int kSideStreams = 16;
constexpr int kPrioLevels = 8, kPoolSlots = 9;
constexpr int kTracePoints = 8;     // CFBPE_PIPE_TRACE: events per sub-batch
#ifndef CFBPE_FRONT_STREAMS
#define CFBPE_FRONT_STREAMS 6
#endif
constexpr int kFrontStreams = CFBPE_FRONT_STREAMS;
constexpr uint64_t kPipeChunkBytes = 12ull << 20;   // largest sub-batch of a pipelined host call (the sizes ramp up to it and down again); measured: profiles/e2e_subbatch_sizes_r01t.jsonl
constexpr uint64_t kPipeMinBytes = 4ull << 20;      // smaller calls run as one shot (a 134 MB batch sharded over 8 GPUs is 16.8 MB a rank: it must still pipeline)

// ---------------------------------------------------------------------------------------
// Structure of a context (SURVEY.md section 8(b): "cfbpe_create(cfg: devices[], n_devices, ...)", "safe to call concurrently from
// several host threads (internal stream pool ...)"):
//   cfbpe_ctx  ->  one DeviceCtx per CUDA device (its copy of every vocabulary's tables, its NCCL communicator)
//              ->  n_workspaces Lanes per device: a Lane is everything ONE call touches on the device -- streams, events, the
//                  workspace, staging buffers, pinned status words -- so calls on different lanes run concurrently.
// A call takes a lane (try-lock round robin, else it waits for one), holds the vocabularies shared (vocab_load holds them
// exclusively) and sets no state outside its lane; the last error is per THREAD.
// A multi-device context shards a host batch by bytes on prompt boundaries, one host thread per device; NCCL (dlopen'ed
// libnccl.so.2: the library links no NCCL symbol) broadcasts the packed tables at vocab load and all-gathers the per-shard
// token totals of every batch, from which each device rebases its offsets (SURVEY.md section 8(e)).
// ---------------------------------------------------------------------------------------
struct Lane {
    std::mutex mu;                        // held for the duration of a call
    int device = 0;
    uint64_t max_bytes = 0;
    cudaStream_t stream = nullptr;       // compute
    cudaStream_t h2d_stream = nullptr;   // pipelined host calls: uploads run ahead of the kernels ...
    cudaStream_t d2h_stream = nullptr;   // ... and downloads trail them
    uint32_t* d_dec_sums = nullptr;      // decode: bytes per tile of kDecodeTile tokens ...
    uint64_t* d_dec_base = nullptr;      // ... and their exclusive scan
    cudaStream_t aux_stream = nullptr;   // the long-piece kernel runs here, next to the short-piece kernel
    cudaStream_t aux2_stream = nullptr;  // ... and the big-piece kernel here, next to both
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
    cudaStream_t side2[kSideStreams] = {};       // pipelined host calls: the big-piece kernel of sub-batch k
    cudaEvent_t ev_list[kMaxPipeChunks] = {};
    cudaEvent_t ev_ws = nullptr;         // recorded at the end of an asynchronous device-path call: the workspace is busy until then
    bool ws_pending = false;             // ... and whether one is outstanding
    uint64_t dev_out_cap = 0;            // out_cap of the last device-path call (cfbpe_device_status reports ENOSPC against it)
    bool dev_want_ids = false;
    cudaEvent_t ev_scan[kMaxPipeChunks] = {};
    cudaStream_t front[kFrontStreams] = {};   // front streams 1.. of a pipelined host call (0 = stream)
    cudaStream_t pool[kPrioLevels][kPoolSlots] = {};   // CFBPE_PIPE_PRIO=1|2 (experiment): streams by priority level
    int prio_mode = 0, prio_levels = 1;
    cudaStream_t side[kSideStreams] = {};  // long-piece tails + emit of sub-batch k overlap the front of k+1
    cudaEvent_t ev_front[kMaxPipeChunks] = {};
    cudaEvent_t ev_h2d[kMaxPipeChunks] = {};
    cudaEvent_t ev_done[kMaxPipeChunks] = {};
    cudaEvent_t ev_chain[kMaxPipeChunks] = {};   // tile_scan of sub-batch k done: the next sub-batch's scan may read tok_end
    cudaEvent_t (*trace)[kTracePoints] = nullptr;           // CFBPE_PIPE_TRACE=1: timed events per sub-batch (h2d, split, short, long, back, d2h) + [nc][0] = start
    DeviceStatus* d_status_arr = nullptr; // one status per sub-batch
    DeviceStatus* h_status_arr = nullptr; // pinned
    uint64_t* h_offs_stage = nullptr;     // pinned: sub-batch-local offsets
    uint64_t* h_totals = nullptr;         // pinned: the all-gathered token totals of a multi-device call [CFBPE_MAX_DEVICES]
    uint64_t* d_totals = nullptr;         // device: the same
    // inputs / outputs of the host API
    uint8_t* d_bytes = nullptr;
    uint64_t* d_offsets = nullptr;
    uint8_t* d_vocab_ids = nullptr;
    uint32_t* d_out_ids = nullptr;
    uint64_t* d_out_offsets = nullptr;
    uint32_t* d_out_counts = nullptr;
    uint32_t* d_budgets = nullptr;        // truncated host calls: per-prompt budgets ...
    uint32_t* d_kept = nullptr;           // ... kept counts ...
    uint64_t* d_cut = nullptr;            // ... and cuts (the rows are staged in d_out_ids)
    Workspace ws{};
    DeviceStatus* h_status = nullptr;  // pinned
    ProfEvents prof{};
};

struct DeviceVocab { uint8_t* d_blob = nullptr; };

struct DeviceCtx {
    int device = 0;
    int index = 0;                        // position in cfbpe_ctx::devs (= NCCL rank)
    int sm_count = 148;
    uint8_t* d_uc1 = nullptr;
    uint8_t* d_uc2 = nullptr;
    uint8_t* d_ascii = nullptr;
    uint16_t* d_fsm = nullptr;
    uint8_t* d_split_tables = nullptr;   // SplitTablesHost: class bytes, 16-wide transition tables, context + product automata (pretok_ctx.h)
    UcTables uc{};
    DeviceVocab vocabs[CFBPE_MAX_VOCABS];
    VocabSet vs{};
    std::vector<std::unique_ptr<Lane>> lanes;
    std::atomic<uint32_t> next_lane{0};
    void* comm = nullptr;                 // ncclComm_t of this device in the context's communicator
};

struct HostVocab { bool loaded = false; std::vector<uint8_t> h_blob; TablesHeader hdr{}; };

// the few NCCL entry points the library uses, resolved at cfbpe_create of a multi-device context
struct NcclApi {
    void* lib = nullptr;
    int (*CommInitAll)(void**, int, const int*) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclChar = 0, kNcclUint64 = 5;       // ncclDataType_t values (nccl.h: ncclInt8 = ncclChar = 0, ncclUint64 = 5)

struct cfbpe_ctx {
    std::vector<std::unique_ptr<DeviceCtx>> devs;
    std::shared_mutex vocab_mu;           // calls: shared; vocabulary load / import: exclusive
    HostVocab vocabs[CFBPE_MAX_VOCABS];
    uint32_t loaded_mask = 0;
    uint64_t max_bytes = 0;
    uint32_t max_prompts = 0;
    uint32_t n_workspaces = 1;
    uint64_t pipe_chunk = kPipeChunkBytes, pipe_min = kPipeMinBytes;   // CFBPE_PIPE_CHUNK_BYTES / CFBPE_PIPE_MIN_BYTES override (tests)
    std::atomic<bool> profiling{false};
    NcclApi nccl;
    bool peer_ok = false;      // several devices, each maps the memory of all the others (NVLink): sub-batches may go round-robin
};

namespace {

// the last error and the last profile are per calling thread: calls run concurrently on one context
thread_local std::string tl_err;
thread_local cfbpe_profile tl_profile{};
thread_local bool tl_profile_ready = false;
thread_local Lane* tl_device_lane = nullptr;      // the lane of this thread's last device-path call (cfbpe_device_status)

// a truncated host call (cfbpe_encode_truncated): the window's parameters and the caller's buffers for its results (counts go
// through the out_counts of the shared path)
struct HostWindow {
    uint32_t max_tokens, keep, pad_id;
    const uint32_t* budgets;   // [n] or nullptr
    uint32_t* rows;            // [n * max_tokens] or nullptr
    uint32_t* kept;            // [n]
    uint64_t* cut;             // [n] or nullptr
};

// the window of the prompts [p0, p0 + n) of a lane's buffers: the rows are staged in d_out_ids at p * L
WindowView lane_window(Lane* ln, const HostWindow& hw, uint32_t p0) {
    return WindowView{hw.max_tokens, hw.keep, hw.pad_id, hw.budgets ? ln->d_budgets + p0 : nullptr,
                      hw.rows ? ln->d_out_ids + static_cast<uint64_t>(p0) * hw.max_tokens : nullptr, ln->d_kept + p0, nullptr,
                      hw.cut ? ln->d_cut + p0 : nullptr};
}
// download the window results of prompts [p0, p0 + n) of a lane (its prompt p0 is the caller's prompt dst0)
cudaError_t download_window(Lane* ln, const HostWindow& hw, uint32_t p0, uint32_t n, uint32_t dst0, cudaStream_t s) {
    if (!n) return cudaSuccess;
    const uint64_t L = hw.max_tokens;
    cudaError_t e = cudaMemcpyAsync(hw.kept + dst0, ln->d_kept + p0, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && hw.cut) e = cudaMemcpyAsync(hw.cut + dst0, ln->d_cut + p0, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && hw.rows) e = cudaMemcpyAsync(hw.rows + dst0 * L, ln->d_out_ids + p0 * L, n * L * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
    return e;
}

int fail(cfbpe_ctx*, int code, const std::string& msg) {
    tl_err = msg;
    return code;
}
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            return fail(ctx, CFBPE_EIO, std::string(#call) + ": " + cudaGetErrorString(e_));             \
        }                                                                                                \
    } while (0)

template <typename T>
cudaError_t dmalloc(T** p, uint64_t count) { return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)); }

// a free lane of the device, locked: round robin without waiting; when all are busy, wait for the next in turn
struct LaneLock {
    Lane* ln = nullptr;
    explicit LaneLock(DeviceCtx* dv) {
        const uint32_t n = static_cast<uint32_t>(dv->lanes.size()), start = dv->next_lane.fetch_add(1);
        for (uint32_t i = 0; i < n && !ln; ++i) { Lane* c = dv->lanes[(start + i) % n].get(); if (c->mu.try_lock()) ln = c; }
        if (!ln) { ln = dv->lanes[start % n].get(); ln->mu.lock(); }
    }
    ~LaneLock() { if (ln) ln->mu.unlock(); }
    LaneLock(const LaneLock&) = delete;
    LaneLock& operator=(const LaneLock&) = delete;
};

int validate_batch(cfbpe_ctx* ctx, uint32_t n, const uint64_t* offsets, const uint8_t* vocab_ids, uint64_t* total_out) {
    if (n > ctx->max_prompts) return fail(ctx, CFBPE_EINVAL, "n_prompts exceeds max_prompts of this context");
    if (!offsets) return fail(ctx, CFBPE_EINVAL, "offsets is NULL");
    if (offsets[0] != 0) return fail(ctx, CFBPE_EINVAL, "offsets[0] must be 0");
    for (uint32_t i = 0; i < n; ++i)
        if (offsets[i + 1] < offsets[i]) return fail(ctx, CFBPE_EINVAL, "offsets are not monotonic at prompt " + std::to_string(i));
    if (offsets[n] > ctx->max_bytes * ctx->devs.size()) return fail(ctx, CFBPE_EINVAL, "batch exceeds max_batch_bytes of this context");
    if (vocab_ids) {
        for (uint32_t i = 0; i < n; ++i)
            if (vocab_ids[i] >= CFBPE_MAX_VOCABS || !ctx->vocabs[vocab_ids[i]].loaded)
                return fail(ctx, CFBPE_ENOENT, "prompt " + std::to_string(i) + " names a vocab that is not loaded");
    } else if (!ctx->vocabs[0].loaded) {
        return fail(ctx, CFBPE_ENOENT, "vocab 0 is not loaded");
    }
    *total_out = offsets[n];
    return CFBPE_OK;
}

// Install a packed table blob as vocabulary vocab_id on EVERY device of the context (caller holds vocab_mu exclusively).
// Device 0 gets it from the host; with several devices the others get it from device 0 by ncclBroadcast over NVLink -- the rank
// file was parsed once, the tables crossed PCIe once.
int install_blob(cfbpe_ctx* ctx, uint32_t vocab_id, std::vector<uint8_t>&& blob) {
    const size_t G = ctx->devs.size();
    std::vector<uint8_t*> nb(G, nullptr);
    auto cleanup = [&]() { for (size_t d = 0; d < G; ++d) { cudaSetDevice(ctx->devs[d]->device); cudaFree(nb[d]); } };
    for (size_t d = 0; d < G; ++d) {
        cudaSetDevice(ctx->devs[d]->device);
        if (cudaMalloc(reinterpret_cast<void**>(&nb[d]), blob.size()) != cudaSuccess) {
            cleanup(); cudaGetLastError();
            return fail(ctx, CFBPE_ENOMEM, "no device memory for the vocabulary tables");
        }
    }
    cudaSetDevice(ctx->devs[0]->device);
    cudaError_t e = cudaMemcpy(nb[0], blob.data(), blob.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cleanup(); return fail(ctx, CFBPE_EIO, std::string("table upload: ") + cudaGetErrorString(e)); }
    if (G > 1) {
        const NcclApi& nc = ctx->nccl;
        int rc = nc.GroupStart();
        for (size_t d = 0; d < G && rc == 0; ++d) {
            cudaSetDevice(ctx->devs[d]->device);
            cudaStream_t st = ctx->devs[d]->lanes[0]->stream;
            rc = nc.Broadcast(nb[0], nb[d], blob.size(), kNcclChar, 0, ctx->devs[d]->comm, st);
        }
        const int rc2 = nc.GroupEnd();
        if (rc == 0) rc = rc2;
        for (size_t d = 0; d < G; ++d) { cudaSetDevice(ctx->devs[d]->device); if (cudaStreamSynchronize(ctx->devs[d]->lanes[0]->stream) != cudaSuccess && rc == 0) rc = -1; }
        if (rc != 0) { cleanup(); return fail(ctx, CFBPE_EIO, std::string("ncclBroadcast of the vocabulary tables: ") + (rc > 0 ? nc.GetErrorString(rc) : "stream error")); }
    }
    HostVocab& hv = ctx->vocabs[vocab_id];
    hv.h_blob = std::move(blob);
    std::memcpy(&hv.hdr, hv.h_blob.data(), sizeof(TablesHeader));
    hv.loaded = true;
    ctx->loaded_mask |= 1u << vocab_id;
    for (size_t d = 0; d < G; ++d) {
        DeviceCtx* dv = ctx->devs[d].get();
        cudaSetDevice(dv->device);
        DeviceVocab& v = dv->vocabs[vocab_id];
        if (v.d_blob) { cudaDeviceSynchronize(); cudaFree(v.d_blob); }   // kernels of a device-path call on any stream may still read the old tables
        v.d_blob = nb[d];
        dv->vs.v[vocab_id] = make_view(v.d_blob, hv.hdr);
        dv->vs.loaded_mask = ctx->loaded_mask;
        // slots that are not loaded alias a loaded one: a bad vocabulary id handed in by a device-path caller is reported
        // (DeviceStatus::bad_vocab -> CFBPE_ENOENT) instead of dereferencing a null table
        for (uint32_t i = 0; i < CFBPE_MAX_VOCABS; ++i) if (!ctx->vocabs[i].loaded) dv->vs.v[i] = dv->vs.v[vocab_id];
    }
    return CFBPE_OK;
}

void fill_profile(Lane* ln, uint64_t n_bytes) {
    cfbpe_profile& p = tl_profile;
    std::memset(&p, 0, sizeof p);
    for (int k = 0; k < CFBPE_NUM_KERNELS; ++k) {
        if (!ln->prof.launched[k]) continue;
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ln->prof.ev[k][0], ln->prof.ev[k][1]) == cudaSuccess) p.kernel_ms[k] = ms;
        p.kernel_launches[k] = (k == K_EMIT) ? 2 : (k == K_WINDOW ? ln->prof.window_launches : 1);   // emit_compact + prompt_offsets
    }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ln->prof.h2d[0], ln->prof.h2d[1]) == cudaSuccess) p.h2d_ms = ms;
    if (cudaEventElapsedTime(&ms, ln->prof.d2h[0], ln->prof.d2h[1]) == cudaSuccess) p.d2h_ms = ms;
    if (cudaEventElapsedTime(&ms, ln->prof.total[0], ln->prof.total[1]) == cudaSuccess) p.total_ms = ms;
    p.n_tokens = ln->h_status->n_tokens;
    p.n_long_pieces = static_cast<uint64_t>(ln->h_status->n_long) + ln->h_status->n_big;
    p.n_bytes = n_bytes;
    p.n_long_bytes = ln->h_status->long_bytes;
    p.n_long_tokens = ln->h_status->long_tokens;
    p.n_miss_pieces = static_cast<uint64_t>(ln->h_status->miss_n[0]) + ln->h_status->miss_n[1] + ln->h_status->miss_n[2];
    p.n_list_pieces = ln->h_status->defer_n;
    p.n_list_parts = ln->h_status->defer_parts;
    p.n_extra_tokens = ln->h_status->extra_n;
    tl_profile_ready = true;
}

// Pipelined host call: the batch is cut into sub-batches of ~kPipeChunkBytes on prompt boundaries; each is an
// independent encode pass on its own slice of the workspace.  Uploads (h2d_stream) run ahead of the kernels
// (stream), downloads (d2h_stream) trail them; token ranks are chained on the device (DeviceStatus::tok_end), so
// ids and offsets land at their final places.  The host only waits for each sub-batch's status to learn how many
// ids to fetch.
// defer != nullptr (a shard of a multi-device call): nothing is downloaded here -- ids, offsets and counts stay in the lane's device
// buffers (dense, shard-local ranks: sub-batch k's offsets at d_out_offsets + p_k + k) and *defer gets the shard's token total.
int run_host_pipelined(cfbpe_ctx* ctx, DeviceCtx* const* dvs, Lane* const* lns, int G, uint32_t n, const uint8_t* bytes, const uint64_t* offsets,
                       const uint8_t* vocab_ids, uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets, uint32_t* out_counts, bool want_ids,
                       uint64_t total, uint64_t* defer, uint32_t* cut_out, int* nc_out, const HostWindow* win) {
    // ---- cut
    uint32_t cut[kMaxPipeChunks + 1];
    const int nc = plan_sub_batches(offsets, n, total, ctx->pipe_chunk, kMaxPipeChunks, cut);
    // Sub-batch k runs on device k mod G (G = 1: the single-device call).  Every device keeps the layout of the whole batch
    // (same slices of its own workspace), so the devices differ only in WHICH sub-batches they fill in; the one thing a sub-batch
    // needs from its predecessor -- the token rank it starts at -- is read from the predecessor's device over NVLink (peer
    // memory), behind a cross-device event.  Uploads and downloads of the devices run side by side on their own PCIe links.
    Lane* ln = lns[0];                       // (host-side staging of the offsets and the trace live in the first lane)
    // local offsets of every sub-batch, staged in pinned memory (sub-batch k occupies [p_k + k, p_{k+1} + k])
    for (int k = 0; k < nc; ++k) {
        const uint32_t p0 = cut[k], p1 = cut[k + 1];
        const uint64_t o0 = offsets[p0];
        uint64_t* dst = ln->h_offs_stage + p0 + k;
        for (uint32_t i = p0; i <= p1; ++i) dst[i - p0] = offsets[i] - o0;
    }
    // ---- enqueue everything that does not depend on the host knowing a result
    const bool trace = G == 1 && getenv("CFBPE_PIPE_TRACE") != nullptr;
    const bool no_copy = trace && getenv("CFBPE_PIPE_NO_COPY") != nullptr;   // measurement aid: the kernels of a pipelined call without its copies (the device buffers still hold the previous call's data)
    if (trace && !ln->trace) {
        ln->trace = new cudaEvent_t[kMaxPipeChunks + 1][kTracePoints];
        for (int k = 0; k <= kMaxPipeChunks; ++k) for (int j = 0; j < kTracePoints; ++j) cudaEventCreate(&ln->trace[k][j]);
    }
    if (trace) CK(cudaEventRecord(ln->trace[nc][0], ln->h2d_stream));
    const auto host_t0 = std::chrono::steady_clock::now();
    auto host_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count(); };
    double host_enq[kMaxPipeChunks] = {}, host_dl[kMaxPipeChunks] = {};
    for (int k = 0; k < nc; ++k) {
        DeviceCtx* const dv = dvs[k % G];
        Lane* const ln = lns[k % G];
        Lane* const prev = k ? lns[(k - 1) % G] : nullptr;
        if (G > 1) CK(cudaSetDevice(dv->device));
        cudaStream_t cs = ln->stream, hs = ln->h2d_stream;
        const uint32_t p0 = cut[k], p1 = cut[k + 1], nk = p1 - p0;
        const uint64_t o0 = offsets[p0], len = offsets[p1] - o0;
        // every sub-batch lands on a 16-byte boundary of the device buffer (K1 reads 16 bytes per lane with one load)
        uint8_t* const d_sub = ln->d_bytes + ((o0 + 15) & ~15ull) + 16ull * k;
        if (len && !no_copy) CK(cudaMemcpyAsync(d_sub, bytes + o0, len, cudaMemcpyHostToDevice, hs));
        CK(cudaMemcpyAsync(ln->d_offsets + p0 + k, lns[0]->h_offs_stage + p0 + k, (static_cast<uint64_t>(nk) + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, hs));
        if (vocab_ids && nk) CK(cudaMemcpyAsync(ln->d_vocab_ids + p0, vocab_ids + p0, nk, cudaMemcpyHostToDevice, hs));
        if (win && win->budgets && nk) CK(cudaMemcpyAsync(ln->d_budgets + p0, win->budgets + p0, nk * sizeof(uint32_t), cudaMemcpyHostToDevice, hs));
        CK(cudaEventRecord(ln->ev_h2d[k], hs));
        if (trace) CK(cudaEventRecord(ln->trace[k][0], hs));
        const int fk = k < kFrontStreams ? k : kFrontStreams - 1;
        cudaStream_t ck = fk ? ln->front[fk] : cs;
        const int lv = ln->prio_mode == 2 ? (k * ln->prio_levels) / nc : 0;
        if (ln->prio_mode) ck = ln->pool[lv][(3 * k + 2) % kPoolSlots];   // the short-piece kernels of sub-batch k: priority falls with k (earlier sub-batches finish, and download, first)
        Workspace w = ln->ws;
        const uint64_t w0 = (o0 >> 5) + 4ull * k;
        w.piece_bits += w0; w.tok_bits += w0; w.pstart_bits += w0;
        w.block_prompt += (o0 >> kPromptBlockShift) + 2ull * k;
        w.dense.by_piece += o0; w.dense.extras += o0; w.dense.extras_cap = static_cast<uint32_t>(len + 1);
        w.dense.tile_pieces += (o0 >> 11) + 2ull * k; w.dense.piece_base += (o0 >> 11) + 2ull * k;
        w.ids_by_pos += o0; w.lscratch.rank += o0; w.lscratch.aux0 += o0; w.lscratch.aux1 += o0;
        w.long_list += (o0 >> 5) + k;
        w.long_cap = static_cast<uint32_t>(len / 32 + 1);
        const uint64_t t0 = (o0 >> 13) + 2ull * k;
        w.tile_counts += t0; w.tile_base += t0;
        w.status = ln->d_status_arr + k;
        w.miss = slice_miss(ln->ws.miss, o0, len, static_cast<uint32_t>(k));
        w.fix_list += (o0 >> 4) + 2ull * k;
        w.fix_cap = static_cast<uint32_t>(len / 16 + 2);
        BatchView b{d_sub, ln->d_offsets + p0 + k, vocab_ids ? ln->d_vocab_ids + p0 : nullptr, nk, len};
        // split, long pieces and the back stage run on a top-priority stream of their own: the long-piece kernels are a latency
        // chain that uses little of the machine, so they start as early as possible and the short-piece kernels fill the rest
        cudaStream_t ss = ln->prio_mode ? ln->pool[lv][(3 * k) % kPoolSlots] : ln->side[k % kSideStreams];
        CK(cudaStreamWaitEvent(ss, ln->ev_h2d[k], 0));
        enqueue_split(b, dv->vs, dv->uc, w, ss, static_cast<ProfEvents*>(nullptr));
        CK(cudaEventRecord(ln->ev_scan[k], ss));
        if (trace) CK(cudaEventRecord(ln->trace[k][1], ss));
        CK(cudaStreamWaitEvent(ck, ln->ev_scan[k], 0));
        cudaStream_t ss2 = ln->prio_mode ? ln->pool[lv][(3 * k + 1) % kPoolSlots] : ln->side2[k % kSideStreams];
        CK(cudaStreamWaitEvent(ss2, ln->ev_scan[k], 0));
        enqueue_list(b, dv->vs, w, static_cast<uint32_t>(dv->sm_count * 4), ss2, static_cast<ProfEvents*>(nullptr));   // the big pieces, beside everything else
        CK(cudaEventRecord(ln->ev_list[k], ss2));
        if (trace) CK(cudaEventRecord(ln->trace[k][6], ss2));
        enqueue_long(b, dv->vs, w, static_cast<uint32_t>(dv->sm_count * 4), ss, static_cast<ProfEvents*>(nullptr));   // tail overlaps what follows on cs
        if (trace) CK(cudaEventRecord(ln->trace[k][3], ss));
        enqueue_short(b, dv->vs, w, static_cast<uint32_t>(dv->sm_count * 4), ck, static_cast<ProfEvents*>(nullptr));
        CK(cudaEventRecord(ln->ev_front[k], ck));
        if (trace) CK(cudaEventRecord(ln->trace[k][2], ck));
        CK(cudaStreamWaitEvent(ss, ln->ev_front[k], 0));
        CK(cudaStreamWaitEvent(ss, ln->ev_list[k], 0));
        enqueue_count(b, w, ss, static_cast<ProfEvents*>(nullptr));
        if (trace) CK(cudaEventRecord(ln->trace[k][7], ss));
        if (k) CK(cudaStreamWaitEvent(ss, prev->ev_chain[k - 1], 0));    // token ranks chain through DeviceStatus::tok_end: only the scan waits
        enqueue_scan(b, w, ss, static_cast<ProfEvents*>(nullptr), k ? &prev->d_status_arr[k - 1].tok_end : nullptr);   // (G > 1: a peer pointer)
        CK(cudaEventRecord(ln->ev_chain[k], ss));
        enqueue_emit(b, w, want_ids ? ln->d_out_ids : nullptr, ctx->max_bytes, ln->d_out_offsets + p0 + k, ln->d_out_counts + p0,
                     ss, static_cast<ProfEvents*>(nullptr));
        if (win) enqueue_window(b, dv->vs, w, ln->d_out_offsets + p0 + k, ln->d_out_counts + p0, lane_window(ln, *win, p0), ss, static_cast<ProfEvents*>(nullptr));
        CK(cudaGetLastError());
        status_publish_kernel<<<1, 64, 0, ss>>>(ln->d_status_arr + k, ln->h_status_arr + k);
        CK(cudaEventRecord(ln->ev_done[k], ss));
        if (trace) { CK(cudaEventRecord(ln->trace[k][4], ss)); host_enq[k] = host_ms(); }
    }
    // ---- trail the kernels with the downloads
    int err = CFBPE_OK;
    uint64_t tok_total = 0;
    for (int k = 0; k < nc; ++k) {
        Lane* const ln = lns[k % G];
        if (G > 1) CK(cudaSetDevice(dvs[k % G]->device));
        cudaStream_t ds = ln->d2h_stream;
        CK(cudaEventSynchronize(ln->ev_done[k]));
        const DeviceStatus st = ln->h_status_arr[k];
        const uint32_t p0 = cut[k], p1 = cut[k + 1], nk = p1 - p0;
        if ((st.long_overflow || st.miss_overflow) && !err) err = fail(ctx, CFBPE_EIO, "internal: long-piece list overflow");
        if (st.bad_vocab && !err) err = fail(ctx, CFBPE_ENOENT, "a prompt names a vocabulary that is not loaded");
        if (st.bad_utf8 && !err) err = fail(ctx, CFBPE_EILSEQ, "a prompt holds malformed UTF-8");
        const uint64_t base = st.tok_end - st.n_tokens;
        tok_total = st.tok_end;
        if (err || defer) continue;
        if (no_copy) continue;
        if (want_ids && st.tok_end <= out_cap && st.n_tokens)
            CK(cudaMemcpyAsync(out_ids + base, ln->d_out_ids + base, st.n_tokens * sizeof(uint32_t), cudaMemcpyDeviceToHost, ds));
        if (out_offsets) CK(cudaMemcpyAsync(out_offsets + p0, ln->d_out_offsets + p0 + k, (static_cast<uint64_t>(nk) + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ds));
        if (out_counts && nk) CK(cudaMemcpyAsync(out_counts + p0, ln->d_out_counts + p0, static_cast<uint64_t>(nk) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ds));
        if (win) CK(download_window(ln, *win, p0, nk, p0, ds));
        if (trace) { CK(cudaEventRecord(ln->trace[k][5], ds)); host_dl[k] = host_ms(); }
    }
    for (int g = 0; g < G; ++g) {
        Lane* const lg = lns[g];
        if (G > 1) CK(cudaSetDevice(dvs[g]->device));
        CK(cudaStreamSynchronize(lg->d2h_stream));
        CK(cudaStreamSynchronize(lg->stream));
        for (int k = 1; k < kFrontStreams; ++k) CK(cudaStreamSynchronize(lg->front[k]));
        for (int k = 0; k < kSideStreams; ++k) CK(cudaStreamSynchronize(lg->side[k]));
        for (int k = 0; k < kSideStreams; ++k) CK(cudaStreamSynchronize(lg->side2[k]));
        if (lg->prio_mode) for (int l = 0; l < kPrioLevels; ++l) for (int j = 0; j < kPoolSlots; ++j) if (lg->pool[l][j]) CK(cudaStreamSynchronize(lg->pool[l][j]));
    }
    if (trace && !err) {
        fprintf(stderr, "pipe trace (ms since the first upload was enqueued): sub-batch bytes | h2d split long_end list_end short count back d2h\n");
        for (int k = 0; k < nc; ++k) {
            float t[kTracePoints] = {};
            for (int j = 0; j < kTracePoints; ++j) if (!(no_copy && j == 5)) cudaEventElapsedTime(&t[j], ln->trace[nc][0], ln->trace[k][j]);
            fprintf(stderr, "  %2d %9llu | %6.2f %6.2f %6.2f %6.2f %6.2f %6.2f %6.2f %6.2f | host: enqueued %.2f download issued %.2f\n", k,
                    static_cast<unsigned long long>(offsets[cut[k + 1]] - offsets[cut[k]]), t[0], t[1], t[3], t[6], t[2], t[7], t[4], t[5], host_enq[k], host_dl[k]);
        }
    }
    if (err) return err;
    if (defer) { *defer = tok_total; if (cut_out) { std::memcpy(cut_out, cut, sizeof(uint32_t) * (nc + 1)); *nc_out = nc; } return CFBPE_OK; }
    if (want_ids && tok_total > out_cap) {
        if (out_offsets) out_offsets[n] = tok_total;
        return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(tok_total) + " ids");
    }
    return CFBPE_OK;
}

// One device's share of a host call (the whole call on a single-device context): validation is done, the lane is locked.
// defer / cut_out / nc_out: see run_host_pipelined; the one-shot path under `defer` leaves everything on the device as ONE sub-batch.
int run_lane(cfbpe_ctx* ctx, DeviceCtx* dv, Lane* ln, uint32_t n, const uint8_t* bytes, const uint64_t* offsets, const uint8_t* vocab_ids,
             uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets, uint32_t* out_counts, bool want_ids, uint64_t total,
             uint64_t* defer = nullptr, uint32_t* cut_out = nullptr, int* nc_out = nullptr, const HostWindow* win = nullptr) {
    CK(cudaSetDevice(dv->device));
    if (ln->ws_pending) { CK(cudaEventSynchronize(ln->ev_ws)); ln->ws_pending = false; }   // an asynchronous device-path call still owns the workspace
    const bool profiling = ctx->profiling.load();
    if (!profiling && total >= ctx->pipe_min && n >= 2)
        return run_host_pipelined(ctx, &dv, &ln, 1, n, bytes, offsets, vocab_ids, out_ids, out_cap, out_offsets, out_counts, want_ids, total, defer, cut_out, nc_out, win);
    cudaStream_t s = ln->stream;
    ProfEvents* prof = profiling ? &ln->prof : nullptr;
    if (prof) { std::memset(prof->launched, 0, sizeof prof->launched); cudaEventRecord(prof->total[0], s); cudaEventRecord(prof->h2d[0], s); }
    if (total) CK(cudaMemcpyAsync(ln->d_bytes, bytes, total, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ln->d_offsets, offsets, (static_cast<uint64_t>(n) + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (vocab_ids && n) CK(cudaMemcpyAsync(ln->d_vocab_ids, vocab_ids, n, cudaMemcpyHostToDevice, s));
    if (win && win->budgets && n) CK(cudaMemcpyAsync(ln->d_budgets, win->budgets, static_cast<uint64_t>(n) * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    if (prof) cudaEventRecord(prof->h2d[1], s);

    BatchView b{ln->d_bytes, ln->d_offsets, vocab_ids ? ln->d_vocab_ids : nullptr, n, total};
    enqueue_encode(b, dv->vs, dv->uc, ln->ws, want_ids ? ln->d_out_ids : nullptr, ctx->max_bytes, ln->d_out_offsets,
                   ln->d_out_counts, static_cast<uint32_t>(dv->sm_count * 4), s, prof ? s : ln->aux_stream, prof ? s : ln->aux2_stream,
                   ln->ev_fork, ln->ev_join, ln->ev_join2, prof);
    if (win) {
        enqueue_window(b, dv->vs, ln->ws, ln->d_out_offsets, ln->d_out_counts, lane_window(ln, *win, 0), s, prof);
        if (prof) prof->window_launches = (win->rows && total) ? 2 : 1;
    }
    CK(cudaGetLastError());
    if (prof) cudaEventRecord(prof->d2h[0], s);
    CK(cudaMemcpyAsync(ln->h_status, ln->ws.status, sizeof(DeviceStatus), cudaMemcpyDeviceToHost, s));
    if (!defer) {
        if (out_offsets) CK(cudaMemcpyAsync(out_offsets, ln->d_out_offsets, (static_cast<uint64_t>(n) + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        if (out_counts && n) CK(cudaMemcpyAsync(out_counts, ln->d_out_counts, static_cast<uint64_t>(n) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        if (win) CK(download_window(ln, *win, 0, n, 0, s));
    }
    CK(cudaStreamSynchronize(s));
    const DeviceStatus st = *ln->h_status;
    if (st.long_overflow || st.miss_overflow) return fail(ctx, CFBPE_EIO, "internal: long-piece list overflow");
    if (st.bad_vocab) return fail(ctx, CFBPE_ENOENT, "a prompt names a vocabulary that is not loaded");
    if (st.bad_utf8) return fail(ctx, CFBPE_EILSEQ, "a prompt holds malformed UTF-8");
    if (defer) { *defer = st.n_tokens; if (cut_out) { cut_out[0] = 0; cut_out[1] = n; *nc_out = 1; } return CFBPE_OK; }
    if (want_ids) {
        if (st.n_tokens > out_cap) {
            if (out_offsets) out_offsets[n] = st.n_tokens;
            return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(st.n_tokens) + " ids");
        }
        if (st.n_tokens) CK(cudaMemcpyAsync(out_ids, ln->d_out_ids, st.n_tokens * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    if (prof) { cudaEventRecord(prof->d2h[1], s); cudaEventRecord(prof->total[1], s); }
    CK(cudaStreamSynchronize(s));
    if (prof) fill_profile(ln, total);
    return CFBPE_OK;
}

// offsets of a shard are ranks inside the shard: add the tokens of the shards before it (the all-gathered totals)
__global__ void rebase_offsets_kernel(uint64_t* __restrict__ offsets, uint64_t n, const uint64_t* __restrict__ totals, uint32_t shard) {
    uint64_t base = 0;
    for (uint32_t d = 0; d < shard; ++d) base += totals[d];
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) offsets[i] += base;
}

// A host call on a multi-device context: the batch is cut into one contiguous range of whole prompts per device, balanced by
// bytes; every device runs its shard on its own host thread and lane (uploads, kernels), the per-shard token totals are
// all-gathered with NCCL (8 bytes a device: the path's only exchange), every device rebases its offsets by the totals of the
// shards before it and downloads ids, offsets and counts straight to their final places in the caller's buffers.
int run_multi_device(cfbpe_ctx* ctx, uint32_t n, const uint8_t* bytes, const uint64_t* offsets, const uint8_t* vocab_ids,
                     uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets, uint32_t* out_counts, bool want_ids, uint64_t total,
                     const HostWindow* win) {
    const uint32_t G = static_cast<uint32_t>(ctx->devs.size());
    std::vector<uint32_t> lo(G + 1, 0);
    for (uint32_t d = 1; d < G; ++d) {      // first prompt whose start is >= d * total / G
        const uint64_t target = total / G * d;
        uint32_t a = lo[d - 1], b = n;
        while (a < b) { const uint32_t m = a + (b - a) / 2; if (offsets[m] >= target) b = m; else a = m + 1; }
        lo[d] = a;
    }
    lo[G] = n;
    for (uint32_t d = 0; d < G; ++d)
        if (offsets[lo[d + 1]] - offsets[lo[d]] > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "a device's shard exceeds max_batch_bytes (one prompt is too large to balance)");
    struct Shard { int rc = CFBPE_OK; std::string err; uint64_t tokens = 0; std::vector<uint64_t> local_offs; uint32_t cut[kMaxPipeChunks + 1]; int nc = 0; };
    std::vector<Shard> sh(G);
    std::vector<std::unique_ptr<LaneLock>> locks(G);
    for (uint32_t d = 0; d < G; ++d) locks[d].reset(new LaneLock(ctx->devs[d].get()));
    // ---- phase 1: every device encodes its shard; results stay on the device
    {
        std::vector<std::thread> th;
        for (uint32_t d = 0; d < G; ++d) th.emplace_back([&, d]() {
            Shard& s = sh[d];
            const uint32_t p0 = lo[d], nd = lo[d + 1] - lo[d];
            const uint64_t o0 = offsets[p0];
            s.local_offs.resize(static_cast<size_t>(nd) + 1);
            for (uint32_t i = 0; i <= nd; ++i) s.local_offs[i] = offsets[p0 + i] - o0;
            HostWindow sw{};                    // (a shard's budgets start at its first prompt; its results are downloaded in phase 2)
            if (win) { sw = *win; if (sw.budgets) sw.budgets += p0; }
            s.rc = run_lane(ctx, ctx->devs[d].get(), locks[d]->ln, nd, bytes + o0, s.local_offs.data(), vocab_ids ? vocab_ids + p0 : nullptr,
                            nullptr, 0, nullptr, nullptr, want_ids, s.local_offs[nd], &s.tokens, s.cut, &s.nc, win ? &sw : nullptr);
            if (s.rc) s.err = tl_err;
        });
        for (auto& t : th) t.join();
    }
    for (uint32_t d = 0; d < G; ++d) if (sh[d].rc) return fail(ctx, sh[d].rc, sh[d].err);
    // ---- phase 2: all-gather of the token totals (NCCL, 8 bytes a device), rebase, download to the final places
    const NcclApi& nc = ctx->nccl;
    int nrc = nc.GroupStart();
    for (uint32_t d = 0; d < G && nrc == 0; ++d) {
        Lane* ln = locks[d]->ln;
        cudaSetDevice(ctx->devs[d]->device);
        ln->h_totals[CFBPE_MAX_DEVICES] = sh[d].tokens;                                   // (slot past the gathered ones: this shard's own total)
        cudaMemcpyAsync(ln->d_totals + CFBPE_MAX_DEVICES, ln->h_totals + CFBPE_MAX_DEVICES, sizeof(uint64_t), cudaMemcpyHostToDevice, ln->stream);
        nrc = nc.AllGather(ln->d_totals + CFBPE_MAX_DEVICES, ln->d_totals, 1, kNcclUint64, ctx->devs[d]->comm, ln->stream);
    }
    { const int r2 = nc.GroupEnd(); if (nrc == 0) nrc = r2; }
    if (nrc != 0) return fail(ctx, CFBPE_EIO, std::string("ncclAllGather of the shard totals: ") + nc.GetErrorString(nrc));
    std::vector<int> rcs(G, CFBPE_OK);
    std::vector<std::string> errs(G);
    uint64_t grand = 0;
    for (uint32_t d = 0; d < G; ++d) grand += sh[d].tokens;
    const bool fits = !want_ids || grand <= out_cap;
    {
        std::vector<std::thread> th;
        for (uint32_t d = 0; d < G; ++d) th.emplace_back([&, d]() {
            Lane* ln = locks[d]->ln;
            const Shard& s = sh[d];
            const uint32_t p0 = lo[d];
            auto ck = [&](cudaError_t e, const char* what) { if (e != cudaSuccess && rcs[d] == CFBPE_OK) { rcs[d] = CFBPE_EIO; errs[d] = std::string(what) + ": " + cudaGetErrorString(e); } };
            ck(cudaSetDevice(ctx->devs[d]->device), "cudaSetDevice");
            cudaStream_t st = ln->stream;
            ck(cudaMemcpyAsync(ln->h_totals, ln->d_totals, sizeof(uint64_t) * G, cudaMemcpyDeviceToHost, st), "totals download");
            for (int k = 0; k < s.nc; ++k) {     // sub-batch k's offsets sit at d_out_offsets + cut[k] + k (run_host_pipelined)
                const uint32_t q0 = s.cut[k], nk = s.cut[k + 1] - s.cut[k];
                const bool last = (k + 1 == s.nc) && (d + 1 == G);
                const uint64_t cnt = static_cast<uint64_t>(nk) + (last ? 1 : 0);      // the boundary entry belongs to the next sub-batch / shard
                if (!cnt) continue;
                uint64_t* src = ln->d_out_offsets + q0 + (s.nc > 1 ? k : 0);
                rebase_offsets_kernel<<<static_cast<unsigned>((cnt + 255) / 256), 256, 0, st>>>(src, cnt, ln->d_totals, d);
                if (out_offsets) ck(cudaMemcpyAsync(out_offsets + p0 + q0, src, cnt * sizeof(uint64_t), cudaMemcpyDeviceToHost, st), "offsets download");
                if (out_counts && nk) ck(cudaMemcpyAsync(out_counts + p0 + q0, ln->d_out_counts + q0, static_cast<uint64_t>(nk) * sizeof(uint32_t), cudaMemcpyDeviceToHost, st), "counts download");
            }
            if (win) ck(download_window(ln, *win, 0, lo[d + 1] - p0, p0, st), "window download");   // rows, kept counts, cuts: prompt-indexed, no rebase
            ck(cudaStreamSynchronize(st), "stream sync");
            uint64_t base = 0;
            for (uint32_t e = 0; e < d; ++e) base += ln->h_totals[e];
            if (want_ids && fits && s.tokens) ck(cudaMemcpyAsync(out_ids + base, ln->d_out_ids, s.tokens * sizeof(uint32_t), cudaMemcpyDeviceToHost, st), "ids download");
            ck(cudaStreamSynchronize(st), "stream sync");
        });
        for (auto& t : th) t.join();
    }
    for (uint32_t d = 0; d < G; ++d) if (rcs[d]) return fail(ctx, rcs[d], errs[d]);
    if (!fits) {
        if (out_offsets) out_offsets[n] = grand;
        return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(grand) + " ids");
    }
    return CFBPE_OK;
}

// shared body of encode_batch / count_batch (host buffers)
int run_host(cfbpe_ctx* ctx, uint32_t n, const uint8_t* bytes, const uint64_t* offsets, const uint8_t* vocab_ids,
             uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets, uint32_t* out_counts, bool want_ids, const HostWindow* win = nullptr) {
    tl_err.clear();
    std::shared_lock<std::shared_mutex> vocabs(ctx->vocab_mu);
    uint64_t total = 0;
    int rc = validate_batch(ctx, n, offsets, vocab_ids, &total);
    if (rc) return rc;
    if (total && !bytes) return fail(ctx, CFBPE_EINVAL, "bytes is NULL");
    if (want_ids && (!out_offsets || (!out_ids && out_cap))) return fail(ctx, CFBPE_EINVAL, "output pointer is NULL");
    if (ctx->devs.size() > 1 && n >= ctx->devs.size() && !ctx->profiling.load()) {
        // Two ways over several devices.  When every device can hold the whole batch (and the devices see each other's memory):
        // the sub-batches of ONE pipelined call go round-robin over the devices -- uploads, kernels and downloads of all devices
        // overlap, the token-rank chain crosses NVLink.  Else: one contiguous shard a device, totals by ncclAllGather.
        if (ctx->peer_ok && total <= ctx->max_bytes && total >= ctx->pipe_min) {
            const int G = static_cast<int>(ctx->devs.size());
            std::vector<std::unique_ptr<LaneLock>> locks(G);
            DeviceCtx* dvs[CFBPE_MAX_DEVICES]; Lane* lns[CFBPE_MAX_DEVICES];
            for (int g = 0; g < G; ++g) {
                dvs[g] = ctx->devs[g].get();
                locks[g].reset(new LaneLock(dvs[g]));
                lns[g] = locks[g]->ln;
                if (lns[g]->ws_pending) { CK(cudaSetDevice(dvs[g]->device)); CK(cudaEventSynchronize(lns[g]->ev_ws)); lns[g]->ws_pending = false; }
            }
            return run_host_pipelined(ctx, dvs, lns, G, n, bytes, offsets, vocab_ids, out_ids, out_cap, out_offsets, out_counts, want_ids, total, nullptr, nullptr, nullptr, win);
        }
        return run_multi_device(ctx, n, bytes, offsets, vocab_ids, out_ids, out_cap, out_offsets, out_counts, want_ids, total, win);
    }
    if (total > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "batch exceeds max_batch_bytes of this context");
    DeviceCtx* dv = ctx->devs[0].get();
    LaneLock lk(dv);
    return run_lane(ctx, dv, lk.ln, n, bytes, offsets, vocab_ids, out_ids, out_cap, out_offsets, out_counts, want_ids, total, nullptr, nullptr, nullptr, win);
}

// ---------------------------------------------------------------------------------------
// construction / destruction
// ---------------------------------------------------------------------------------------
void destroy_lane(Lane* ln) {
    if (!ln) return;
    cudaSetDevice(ln->device);
    cudaFree(ln->d_bytes); cudaFree(ln->d_offsets); cudaFree(ln->d_vocab_ids);
    cudaFree(ln->d_out_ids); cudaFree(ln->d_out_offsets); cudaFree(ln->d_out_counts);
    cudaFree(ln->d_budgets); cudaFree(ln->d_kept); cudaFree(ln->d_cut);
    cudaFree(ln->ws.piece_bits); cudaFree(ln->ws.tok_bits); cudaFree(ln->ws.ids_by_pos);
    cudaFree(ln->ws.lscratch.rank); cudaFree(ln->ws.lscratch.aux0); cudaFree(ln->ws.lscratch.aux1);
    for (uint32_t c = 0; c < 3; ++c) cudaFree(ln->ws.miss.list[c]);
    cudaFree(ln->d_dec_sums); cudaFree(ln->d_dec_base); cudaFree(ln->d_totals);
    cudaFree(ln->ws.dense.by_piece); cudaFree(ln->ws.dense.extras); cudaFree(ln->ws.dense.tile_pieces); cudaFree(ln->ws.dense.piece_base);
    cudaFree(ln->ws.fix_list); cudaFree(ln->ws.pstart_bits); cudaFree(ln->ws.block_prompt);
    cudaFree(ln->ws.long_list); cudaFree(ln->ws.tile_counts); cudaFree(ln->ws.tile_base); cudaFree(ln->ws.status);
    if (ln->h_status) cudaFreeHost(ln->h_status);
    if (ln->h_status_arr) cudaFreeHost(ln->h_status_arr);
    if (ln->h_offs_stage) cudaFreeHost(ln->h_offs_stage);
    if (ln->h_totals) cudaFreeHost(ln->h_totals);
    cudaFree(ln->d_status_arr);
    for (int k = 0; k < kMaxPipeChunks; ++k) {
        if (ln->ev_h2d[k]) cudaEventDestroy(ln->ev_h2d[k]); if (ln->ev_done[k]) cudaEventDestroy(ln->ev_done[k]);
        if (ln->ev_front[k]) cudaEventDestroy(ln->ev_front[k]); if (ln->ev_chain[k]) cudaEventDestroy(ln->ev_chain[k]);
        if (ln->ev_scan[k]) cudaEventDestroy(ln->ev_scan[k]); if (ln->ev_list[k]) cudaEventDestroy(ln->ev_list[k]);
    }
    for (int k = 1; k < kFrontStreams; ++k) if (ln->front[k]) cudaStreamDestroy(ln->front[k]);
    for (int l = 0; l < kPrioLevels; ++l) for (int j = 0; j < kPoolSlots; ++j) if (ln->pool[l][j]) cudaStreamDestroy(ln->pool[l][j]);
    for (int k = 0; k < kSideStreams; ++k) { if (ln->side[k]) cudaStreamDestroy(ln->side[k]); if (ln->side2[k]) cudaStreamDestroy(ln->side2[k]); }
    if (ln->aux_stream) cudaStreamDestroy(ln->aux_stream);
    if (ln->aux2_stream) cudaStreamDestroy(ln->aux2_stream);
    if (ln->ev_fork) cudaEventDestroy(ln->ev_fork);
    if (ln->ev_join) cudaEventDestroy(ln->ev_join);
    if (ln->ev_join2) cudaEventDestroy(ln->ev_join2);
    if (ln->ev_ws) cudaEventDestroy(ln->ev_ws);
    if (ln->h2d_stream) cudaStreamDestroy(ln->h2d_stream);
    if (ln->d2h_stream) cudaStreamDestroy(ln->d2h_stream);
    for (int k = 0; k < CFBPE_NUM_KERNELS; ++k) for (int j = 0; j < 2; ++j) if (ln->prof.ev[k][j]) cudaEventDestroy(ln->prof.ev[k][j]);
    for (int j = 0; j < 2; ++j) {
        if (ln->prof.h2d[j]) cudaEventDestroy(ln->prof.h2d[j]);
        if (ln->prof.d2h[j]) cudaEventDestroy(ln->prof.d2h[j]);
        if (ln->prof.total[j]) cudaEventDestroy(ln->prof.total[j]);
    }
    if (ln->stream) cudaStreamDestroy(ln->stream);
}

// everything one call touches on the device, sized by max_batch_bytes (~33 bytes per byte of it)
bool create_lane(Lane* ln, int device, uint64_t mb, uint64_t mp) {
    ln->device = device;
    ln->max_bytes = mb;
    const uint64_t nw = n_flag_words(mb) + 4 + 4 * kMaxPipeChunks;      // + per-sub-batch slack of a pipelined call
    const uint64_t nt = n_scan_tiles(mb) + 1 + 2 * kMaxPipeChunks;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    bool ok = cudaStreamCreateWithPriority(&ln->stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;   // front stream of sub-batch 0
    ok = ok && dmalloc(&ln->d_bytes, mb + 256 + 16 * (kMaxPipeChunks + 1)) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_offsets, mp + 1 + kMaxPipeChunks) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_vocab_ids, mp + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_out_ids, mb + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_out_offsets, mp + 1 + kMaxPipeChunks) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_out_counts, mp + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_budgets, mp + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_kept, mp + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_cut, mp + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.piece_bits, nw) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.tok_bits, nw) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.ids_by_pos, mb + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.lscratch.rank, mb + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.lscratch.aux0, mb + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.lscratch.aux1, mb + 1) == cudaSuccess;
    ln->ws.long_cap = static_cast<uint32_t>(mb / 32 + 1 + kMaxPipeChunks);   // a long piece holds more than 32 bytes
    ok = ok && dmalloc(&ln->ws.long_list, ln->ws.long_cap) == cudaSuccess;
    for (uint32_t c = 0; c < 3; ++c) {
        const uint64_t words = miss_list_words(mb, c, kMaxPipeChunks);      // 64-bit entries
        ok = ok && dmalloc(&ln->ws.miss.list[c], words) == cudaSuccess;
        ln->ws.miss.cap[c] = static_cast<uint32_t>(words);
    }
    ok = ok && dmalloc(&ln->ws.dense.by_piece, mb + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.dense.extras, mb + 1) == cudaSuccess;
    ln->ws.dense.extras_cap = static_cast<uint32_t>(mb + 1);
    ok = ok && dmalloc(&ln->ws.dense.tile_pieces, (mb >> 11) + 2 + 2 * kMaxPipeChunks) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.dense.piece_base, (mb >> 11) + 2 + 2 * kMaxPipeChunks) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.pstart_bits, nw) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.block_prompt, (mb >> kPromptBlockShift) + 2 + 2 * kMaxPipeChunks) == cudaSuccess;
    ln->ws.fix_cap = static_cast<uint32_t>(mb / 16 + 2 + 2 * kMaxPipeChunks);
    ok = ok && dmalloc(&ln->ws.fix_list, ln->ws.fix_cap) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_dec_sums, mb / kDecodeTile + 2) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_dec_base, mb / kDecodeTile + 2) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_totals, CFBPE_MAX_DEVICES + 1) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.tile_counts, nt) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.tile_base, nt) == cudaSuccess;
    ok = ok && dmalloc(&ln->ws.status, 1) == cudaSuccess;
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&ln->h_status), sizeof(DeviceStatus)) == cudaSuccess;
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&ln->h_totals), sizeof(uint64_t) * (CFBPE_MAX_DEVICES + 1)) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ln->h2d_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ln->d2h_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && dmalloc(&ln->d_status_arr, kMaxPipeChunks) == cudaSuccess;
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&ln->h_status_arr), sizeof(DeviceStatus) * kMaxPipeChunks) == cudaSuccess;
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&ln->h_offs_stage), sizeof(uint64_t) * (mp + 1 + kMaxPipeChunks)) == cudaSuccess;
    {   // a pipelined host call gives earlier sub-batches the higher priority, so that they finish first and their downloads
        // run while the later ones compute (with equal priorities the sub-batches finished together and the downloads queued up
        // at the end: tools/pipe_trace.py)
        const int levels = prio_lo - prio_hi + 1;
        for (int k = 1; ok && k < kFrontStreams; ++k)
            ok = cudaStreamCreateWithPriority(&ln->front[k], cudaStreamNonBlocking, prio_hi + (k < levels ? k : levels - 1)) == cudaSuccess;
        for (int k = 0; ok && k < kSideStreams; ++k) ok = cudaStreamCreateWithPriority(&ln->side[k], cudaStreamNonBlocking, prio_hi) == cudaSuccess;
        for (int k = 0; ok && k < kSideStreams; ++k) ok = cudaStreamCreateWithPriority(&ln->side2[k], cudaStreamNonBlocking, prio_hi) == cudaSuccess;
        if (const char* e = std::getenv("CFBPE_PIPE_PRIO")) {      // experiment: 1 = every kernel at one priority, 2 = priority by the sub-batch's age
            ln->prio_mode = std::atoi(e);
            ln->prio_levels = ln->prio_mode == 2 ? (levels < kPrioLevels ? levels : kPrioLevels) : 1;
            for (int l = 0; ok && ln->prio_mode && l < ln->prio_levels; ++l)
                for (int j = 0; ok && j < kPoolSlots; ++j) ok = cudaStreamCreateWithPriority(&ln->pool[l][j], cudaStreamNonBlocking, prio_hi + l) == cudaSuccess;
        }
    }
    // the long-piece kernels are latency-bound and small: their CTAs go first, the short-piece kernels fill the rest
    // (A/B of lower priorities and of CTA caps: no gain, profiles/ab_bench_r02h.txt)
    ok = ok && cudaStreamCreateWithPriority(&ln->aux_stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    ok = ok && cudaStreamCreateWithPriority(&ln->aux2_stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ln->ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&ln->ev_join, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ln->ev_ws, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ln->ev_join2, cudaEventDisableTiming) == cudaSuccess;
    for (int k = 0; ok && k < kMaxPipeChunks; ++k)
        ok = cudaEventCreateWithFlags(&ln->ev_h2d[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ln->ev_front[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ln->ev_done[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ln->ev_chain[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ln->ev_scan[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ln->ev_list[k], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMemset(ln->d_bytes, 0, mb + 256 + 16 * (kMaxPipeChunks + 1)) == cudaSuccess;
    for (int k = 0; ok && k < CFBPE_NUM_KERNELS; ++k)
        ok = cudaEventCreate(&ln->prof.ev[k][0]) == cudaSuccess && cudaEventCreate(&ln->prof.ev[k][1]) == cudaSuccess;
    for (int k = 0; ok && k < 2; ++k)
        ok = cudaEventCreate(&ln->prof.h2d[k]) == cudaSuccess && cudaEventCreate(&ln->prof.d2h[k]) == cudaSuccess &&
             cudaEventCreate(&ln->prof.total[k]) == cudaSuccess;
    return ok;
}

bool create_device(DeviceCtx* dv, int device, int index, uint32_t n_lanes, uint64_t mb, uint64_t mp) {
    dv->device = device; dv->index = index;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) return false;     // sm_100a SASS only
    if (cudaSetDevice(device) != cudaSuccess) return false;
    dv->sm_count = prop.multiProcessorCount;
    bool ok = cudaFuncSetAttribute(bpe_list_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kListSmemBytes)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(pretok_split16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kNumPatterns * kProdTableBytes)) == cudaSuccess;
    ok = ok && dmalloc(&dv->d_uc1, sizeof cfbpe_uc_stage1) == cudaSuccess;
    ok = ok && dmalloc(&dv->d_uc2, sizeof cfbpe_uc_stage2) == cudaSuccess;
    ok = ok && cudaMemcpy(dv->d_uc1, cfbpe_uc_stage1, sizeof cfbpe_uc_stage1, cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(dv->d_uc2, cfbpe_uc_stage2, sizeof cfbpe_uc_stage2, cudaMemcpyHostToDevice) == cudaSuccess;
    {
        std::vector<uint16_t> fsm(kNumPatterns * kPretokTableSize);
        uint8_t ascii[128];
        build_pretok_tables(fsm.data());
        build_ascii_classes(ascii);
        ok = ok && dmalloc(&dv->d_ascii, 128) == cudaSuccess;
        ok = ok && dmalloc(&dv->d_fsm, fsm.size()) == cudaSuccess;
        ok = ok && cudaMemcpy(dv->d_ascii, ascii, 128, cudaMemcpyHostToDevice) == cudaSuccess;
        ok = ok && cudaMemcpy(dv->d_fsm, fsm.data(), fsm.size() * sizeof(uint16_t), cudaMemcpyHostToDevice) == cudaSuccess;
        std::vector<SplitTablesHost> st(1);
        build_split_tables(st.data());
        ok = ok && dmalloc(&dv->d_split_tables, sizeof(SplitTablesHost)) == cudaSuccess;
        ok = ok && cudaMemcpy(dv->d_split_tables, st.data(), sizeof(SplitTablesHost), cudaMemcpyHostToDevice) == cudaSuccess;
    }
    if (!ok) return false;
    dv->uc = UcTables{dv->d_uc1, dv->d_uc2, dv->d_ascii, dv->d_fsm,
                      dv->d_split_tables + offsetof(SplitTablesHost, cls256),
                      reinterpret_cast<const uint16_t*>(dv->d_split_tables + offsetof(SplitTablesHost, fsm16)),
                      reinterpret_cast<const uint16_t*>(dv->d_split_tables + offsetof(SplitTablesHost, ctx16)),
                      reinterpret_cast<const uint64_t*>(dv->d_split_tables + offsetof(SplitTablesHost, prod)),
                      reinterpret_cast<const ProdInfo*>(dv->d_split_tables + offsetof(SplitTablesHost, prod_info)),
                      dv->d_split_tables + offsetof(SplitTablesHost, prod_skip),
                      dv->d_split_tables + offsetof(SplitTablesHost, prod_start)};
    for (uint32_t i = 0; i < n_lanes; ++i) {
        dv->lanes.emplace_back(new Lane());
        if (!create_lane(dv->lanes.back().get(), device, mb, mp)) return false;
    }
    return true;
}

bool load_nccl(NcclApi* n) {
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) { n->lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (n->lib) break; }
    if (!n->lib) return false;
    auto sym = [&](const char* s) { return dlsym(n->lib, s); };
    n->CommInitAll = reinterpret_cast<decltype(n->CommInitAll)>(sym("ncclCommInitAll"));
    n->CommDestroy = reinterpret_cast<decltype(n->CommDestroy)>(sym("ncclCommDestroy"));
    n->GroupStart = reinterpret_cast<decltype(n->GroupStart)>(sym("ncclGroupStart"));
    n->GroupEnd = reinterpret_cast<decltype(n->GroupEnd)>(sym("ncclGroupEnd"));
    n->Broadcast = reinterpret_cast<decltype(n->Broadcast)>(sym("ncclBroadcast"));
    n->AllGather = reinterpret_cast<decltype(n->AllGather)>(sym("ncclAllGather"));
    n->GetErrorString = reinterpret_cast<decltype(n->GetErrorString)>(sym("ncclGetErrorString"));
    return n->CommInitAll && n->CommDestroy && n->GroupStart && n->GroupEnd && n->Broadcast && n->AllGather && n->GetErrorString;
}

}  // namespace

// Every entry point that selects a device puts the caller's current device back on return: the library is a guest in the host
// process (a model runtime next door expects its own device to stay current on its thread).
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

extern "C" {

int cfbpe_abi_version(void) { return static_cast<int>(CFBPE_ABI_VERSION); }

#ifndef CFBPE_SRC_HASH
#define CFBPE_SRC_HASH "unknown"
#endif
const char* cfbpe_build_id(void) { return CFBPE_SRC_HASH; }

int cfbpe_create(const cfbpe_config* cfg, cfbpe_ctx** out) {
    DeviceGuard restore_device;
    if (!cfg || !out || cfg->struct_size < offsetof(cfbpe_config, devices)) return CFBPE_EINVAL;
    *out = nullptr;
    // (a pipelined host call keeps ~20 streams busy: hosts should export CUDA_DEVICE_MAX_CONNECTIONS=32 before CUDA
    //  initialises -- INTEGRATION.md; the library does not touch the process environment)
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return CFBPE_ENODEV;
    // the fields after `flags` exist when the caller's struct is new enough (struct_size versions the struct)
    const bool has_multi = cfg->struct_size >= sizeof(cfbpe_config);
    std::vector<int> devices;
    if (has_multi && cfg->n_devices > 0) {
        if (cfg->n_devices > CFBPE_MAX_DEVICES) return CFBPE_EINVAL;
        for (uint32_t i = 0; i < cfg->n_devices; ++i) devices.push_back(cfg->devices[i]);
    } else devices.push_back(cfg->device);
    for (size_t i = 0; i < devices.size(); ++i) {
        if (devices[i] < 0 || devices[i] >= ndev) return CFBPE_ENODEV;
        for (size_t j = 0; j < i; ++j) if (devices[j] == devices[i]) return CFBPE_EINVAL;
    }
    cfbpe_ctx* ctx = new (std::nothrow) cfbpe_ctx();
    if (!ctx) return CFBPE_ENOMEM;
    ctx->max_bytes = cfg->max_batch_bytes ? cfg->max_batch_bytes : (256ull << 20);
    ctx->max_prompts = cfg->max_prompts ? cfg->max_prompts : (1u << 20);
    ctx->n_workspaces = (has_multi && cfg->n_workspaces) ? cfg->n_workspaces : 1u;
    if (ctx->max_bytes >= (1ull << 32) - 4096 || ctx->n_workspaces > 16) { delete ctx; return CFBPE_EINVAL; }   // byte positions inside a batch are 32-bit in the work lists
    if (devices.size() > 1 && !load_nccl(&ctx->nccl)) { delete ctx; tl_err = "a multi-device context needs libnccl.so.2 (vocabulary broadcast, gather of the shard totals)"; return CFBPE_EIO; }
    for (size_t i = 0; i < devices.size(); ++i) {
        ctx->devs.emplace_back(new DeviceCtx());
        if (!create_device(ctx->devs.back().get(), devices[i], static_cast<int>(i), ctx->n_workspaces, ctx->max_bytes, ctx->max_prompts)) {
            const bool nodev = ctx->devs.back()->sm_count == 148 && ctx->devs.back()->lanes.empty() && !ctx->devs.back()->d_uc1;
            cudaGetLastError();
            cfbpe_destroy(ctx);
            return nodev ? CFBPE_ENODEV : CFBPE_ENOMEM;
        }
    }
    if (devices.size() > 1) {
        std::vector<void*> comms(devices.size(), nullptr);
        const int rc = ctx->nccl.CommInitAll(comms.data(), static_cast<int>(devices.size()), devices.data());
        if (rc != 0) { tl_err = std::string("ncclCommInitAll: ") + ctx->nccl.GetErrorString(rc); cfbpe_destroy(ctx); return CFBPE_EIO; }
        for (size_t i = 0; i < devices.size(); ++i) ctx->devs[i]->comm = comms[i];
        // peer mappings: a sub-batch on one device reads the token rank its predecessor on another device ended at
        bool peers = std::getenv("CFBPE_NO_PEER") == nullptr;
        for (size_t a = 0; a < devices.size() && peers; ++a) {
            cudaSetDevice(devices[a]);
            for (size_t b2 = 0; b2 < devices.size() && peers; ++b2) {
                if (a == b2) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, devices[a], devices[b2]) != cudaSuccess || !can) { peers = false; break; }
                const cudaError_t e = cudaDeviceEnablePeerAccess(devices[b2], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) peers = false;
                cudaGetLastError();
            }
        }
        ctx->peer_ok = peers;
    }
    if (const char* e = std::getenv("CFBPE_PIPE_CHUNK_BYTES")) { const uint64_t v = std::strtoull(e, nullptr, 10); if (v >= 1024) ctx->pipe_chunk = v; }
    if (const char* e = std::getenv("CFBPE_PIPE_MIN_BYTES")) { const uint64_t v = std::strtoull(e, nullptr, 10); if (v >= 1) ctx->pipe_min = v; }
    *out = ctx;
    return CFBPE_OK;
}

void cfbpe_destroy(cfbpe_ctx* ctx) {
    DeviceGuard restore_device;
    if (!ctx) return;
    for (auto& dvp : ctx->devs) {
        DeviceCtx* dv = dvp.get();
        cudaSetDevice(dv->device);
        cudaDeviceSynchronize();             // device-path calls may still be running on the caller's streams
        if (dv->comm && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(dv->comm);
        for (auto& ln : dv->lanes) destroy_lane(ln.get());
        cudaSetDevice(dv->device);
        cudaFree(dv->d_uc1); cudaFree(dv->d_uc2); cudaFree(dv->d_ascii); cudaFree(dv->d_fsm); cudaFree(dv->d_split_tables);
        for (auto& v : dv->vocabs) { if (v.d_blob) cudaFree(v.d_blob); }
    }
    delete ctx;
}

const char* cfbpe_last_error(const cfbpe_ctx*) { return tl_err.c_str(); }

int cfbpe_vocab_load(cfbpe_ctx* ctx, uint32_t vocab_id, const uint8_t* ranks_file, size_t len, uint32_t format,
                     uint32_t pattern_id, uint32_t max_ranks) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    if (vocab_id >= CFBPE_MAX_VOCABS) return fail(ctx, CFBPE_EINVAL, "vocab_id out of range");
    if (!ranks_file || !len) return fail(ctx, CFBPE_EINVAL, "empty rank file");
    if (pattern_id >= CFBPE_PATTERN_COUNT) return fail(ctx, CFBPE_EINVAL, "unknown pattern id");
    std::vector<std::string> toks;
    std::string e;
    int rc;
    if (format == CFBPE_FORMAT_TIKTOKEN) rc = parse_tiktoken(ranks_file, len, max_ranks, toks, e);
    else if (format == CFBPE_FORMAT_TEKKEN_JSON) rc = parse_tekken_json(ranks_file, len, max_ranks, toks, e);
    else return fail(ctx, CFBPE_EINVAL, "unknown rank-file format");
    if (rc) return fail(ctx, rc, e);
    std::vector<uint8_t> blob;
    rc = build_tables(toks, pattern_id, blob, e);
    if (rc) return fail(ctx, rc, e);
    std::unique_lock<std::shared_mutex> lock(ctx->vocab_mu);
    return install_blob(ctx, vocab_id, std::move(blob));
}

int cfbpe_vocab_get_info(const cfbpe_ctx* ctx, uint32_t vocab_id, cfbpe_vocab_info* out) {
    if (!ctx || !out || vocab_id >= CFBPE_MAX_VOCABS) return CFBPE_EINVAL;
    const HostVocab& v = ctx->vocabs[vocab_id];
    if (!v.loaded) return CFBPE_ENOENT;
    out->n_ranks = v.hdr.n_ranks;
    out->pattern_id = v.hdr.pattern_id;
    out->max_token_len = v.hdr.max_token_len;
    out->n_pair_entries = v.hdr.n_pair_entries;
    out->table_bytes = v.hdr.total_bytes;
    return CFBPE_OK;
}

int cfbpe_vocab_export(const cfbpe_ctx* ctx, uint32_t vocab_id, uint8_t* buf, uint64_t cap, uint64_t* size) {
    if (!ctx || vocab_id >= CFBPE_MAX_VOCABS) return CFBPE_EINVAL;
    const HostVocab& v = ctx->vocabs[vocab_id];
    if (!v.loaded) return CFBPE_ENOENT;
    if (size) *size = v.h_blob.size();
    if (!buf) return CFBPE_OK;
    if (cap < v.h_blob.size()) return CFBPE_ENOSPC;
    std::memcpy(buf, v.h_blob.data(), v.h_blob.size());
    return CFBPE_OK;
}

int cfbpe_vocab_import(cfbpe_ctx* ctx, uint32_t vocab_id, const uint8_t* buf, uint64_t size) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    if (vocab_id >= CFBPE_MAX_VOCABS || !buf) return fail(ctx, CFBPE_EINVAL, "bad argument");
    std::string e;
    int rc = validate_tables(buf, size, e);
    if (rc) return fail(ctx, rc, e);
    std::unique_lock<std::shared_mutex> lock(ctx->vocab_mu);
    return install_blob(ctx, vocab_id, std::vector<uint8_t>(buf, buf + size));
}

int cfbpe_encode_batch(cfbpe_ctx* ctx, uint32_t n_prompts, const uint8_t* bytes, const uint64_t* offsets,
                       const uint8_t* vocab_ids, uint32_t* out_ids, uint64_t out_cap, uint64_t* out_offsets,
                       uint32_t* out_counts) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    return run_host(ctx, n_prompts, bytes, offsets, vocab_ids, out_ids, out_cap, out_offsets, out_counts, true);
}

int cfbpe_count_batch(cfbpe_ctx* ctx, uint32_t n_prompts, const uint8_t* bytes, const uint64_t* offsets,
                      const uint8_t* vocab_ids, uint32_t* out_counts) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    if (!out_counts && n_prompts) return fail(ctx, CFBPE_EINVAL, "out_counts is NULL");
    return run_host(ctx, n_prompts, bytes, offsets, vocab_ids, nullptr, 0, nullptr, out_counts, false);
}

int cfbpe_encode_truncated(cfbpe_ctx* ctx, uint32_t n_prompts, const uint8_t* bytes, const uint64_t* offsets, const uint8_t* vocab_ids,
                           uint32_t max_tokens, uint32_t keep, uint32_t pad_id, const uint32_t* budgets, uint32_t* out_rows,
                           uint32_t* out_kept, uint32_t* out_counts, uint64_t* out_cut) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    if (!max_tokens) return fail(ctx, CFBPE_EINVAL, "max_tokens must be at least 1");
    if (keep != CFBPE_KEEP_HEAD && keep != CFBPE_KEEP_TAIL) return fail(ctx, CFBPE_EINVAL, "keep must be CFBPE_KEEP_HEAD or CFBPE_KEEP_TAIL");
    if (!out_kept && n_prompts) return fail(ctx, CFBPE_EINVAL, "out_kept is NULL");
    if (out_rows && static_cast<uint64_t>(n_prompts) * max_tokens > ctx->max_bytes)
        return fail(ctx, CFBPE_EINVAL, "n_prompts x max_tokens exceeds max_batch_bytes of this context (the rows are staged in its id buffer)");
    const HostWindow win{max_tokens, keep, pad_id, budgets, out_rows, out_kept, out_cut};
    return run_host(ctx, n_prompts, bytes, offsets, vocab_ids, nullptr, 0, nullptr, out_counts, false, &win);
}

int cfbpe_decode_batch(cfbpe_ctx* ctx, uint32_t n_seqs, const uint32_t* ids, const uint64_t* id_offsets,
                       const uint8_t* vocab_ids, uint8_t* out_bytes, uint64_t out_cap, uint64_t* out_offsets) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    std::shared_lock<std::shared_mutex> vocabs(ctx->vocab_mu);
    if (!id_offsets || !out_offsets) return fail(ctx, CFBPE_EINVAL, "offsets pointer is NULL");
    if (n_seqs > ctx->max_prompts) return fail(ctx, CFBPE_EINVAL, "batch exceeds the limits of this context");
    if (id_offsets[0] != 0) return fail(ctx, CFBPE_EINVAL, "id_offsets[0] must be 0");
    for (uint32_t i = 0; i < n_seqs; ++i) if (id_offsets[i + 1] < id_offsets[i]) return fail(ctx, CFBPE_EINVAL, "id_offsets must not decrease");
    const uint64_t n_ids = id_offsets[n_seqs];
    if (n_ids > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "batch exceeds the limits of this context");
    if (n_ids && !ids) return fail(ctx, CFBPE_EINVAL, "ids is NULL");
    for (uint32_t i = 0; vocab_ids && i < n_seqs; ++i)
        if (vocab_ids[i] >= kMaxVocabs || !ctx->vocabs[vocab_ids[i]].loaded) return fail(ctx, CFBPE_ENOENT, "vocab " + std::to_string(vocab_ids[i]) + " is not loaded");
    if (!vocab_ids && !ctx->vocabs[0].loaded) return fail(ctx, CFBPE_ENOENT, "vocab 0 is not loaded");
    DeviceCtx* dv = ctx->devs[0].get();      // (decode runs on the first device: it is not on the hot path)
    LaneLock lk(dv);
    Lane* ln = lk.ln;
    CK(cudaSetDevice(dv->device));
    if (ln->ws_pending) { CK(cudaEventSynchronize(ln->ev_ws)); ln->ws_pending = false; }
    cudaStream_t s = ln->stream;
    if (n_ids) CK(cudaMemcpyAsync(ln->d_out_ids, ids, n_ids * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ln->d_offsets, id_offsets, (static_cast<uint64_t>(n_seqs) + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (vocab_ids && n_seqs) CK(cudaMemcpyAsync(ln->d_vocab_ids, vocab_ids, n_seqs, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(ln->ws.status, 0, sizeof(DeviceStatus), s));
    DecodeView d{ln->d_out_ids, ln->d_offsets, vocab_ids ? ln->d_vocab_ids : nullptr, n_seqs, n_ids};
    const uint32_t n_tiles = static_cast<uint32_t>((n_ids + kDecodeTile - 1) / kDecodeTile);
    if (n_tiles) decode_len_kernel<<<n_tiles, 256, 0, s>>>(d, dv->vs, ln->ws.ids_by_pos, ln->d_dec_sums, ln->ws.status);
    tile_scan_kernel<<<1, n_tiles ? 1024 : 32, 0, s>>>(ln->d_dec_sums, n_tiles, ln->d_dec_base, ln->ws.status, nullptr);
    if (n_tiles) decode_copy_kernel<<<n_tiles, 256, 0, s>>>(d, dv->vs, ln->ws.ids_by_pos, ln->d_dec_base, ln->d_bytes, ctx->max_bytes);
    decode_offsets_kernel<<<static_cast<unsigned>((static_cast<uint64_t>(n_seqs) + 1 + 255) / 256), 256, 0, s>>>(d, ln->ws.ids_by_pos, ln->d_dec_base, ln->d_out_offsets, ln->ws.status);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ln->h_status, ln->ws.status, sizeof(DeviceStatus), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const DeviceStatus st = *ln->h_status;
    if (st.bad_utf8) return fail(ctx, CFBPE_EINVAL, "a token id is outside its vocabulary");
    const uint64_t total = st.tok_end;
    if (total > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "the decoded batch exceeds max_batch_bytes of this context");
    CK(cudaMemcpyAsync(out_offsets, ln->d_out_offsets, (static_cast<uint64_t>(n_seqs) + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (total > out_cap || (total && !out_bytes)) {
        CK(cudaStreamSynchronize(s));
        out_offsets[n_seqs] = total;
        return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(total) + " bytes");
    }
    if (total) CK(cudaMemcpyAsync(out_bytes, ln->d_bytes, total, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return CFBPE_OK;
}

int cfbpe_encode_batch_device(cfbpe_ctx* ctx, uint32_t n_prompts, const uint8_t* d_bytes, uint64_t total_bytes,
                              const uint64_t* d_offsets, const uint8_t* d_vocab_ids, uint32_t* d_out_ids,
                              uint64_t out_cap, uint64_t* d_out_offsets, uint32_t* d_out_counts, uint64_t* n_tokens,
                              void* stream) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    std::shared_lock<std::shared_mutex> vocabs(ctx->vocab_mu);
    if (n_prompts > ctx->max_prompts || total_bytes > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "batch exceeds the limits of this context");
    if (!d_offsets || !d_out_offsets || (total_bytes && !d_bytes)) return fail(ctx, CFBPE_EINVAL, "device pointer is NULL");
    if (!ctx->vocabs[0].loaded && !d_vocab_ids) return fail(ctx, CFBPE_ENOENT, "vocab 0 is not loaded");
    if (!ctx->loaded_mask) return fail(ctx, CFBPE_ENOENT, "no vocabulary is loaded");
    // the buffers live on ONE device: the first of the context whose ordinal is current, else the first
    DeviceCtx* dv = ctx->devs[0].get();
    { int cur = -1; if (cudaGetDevice(&cur) == cudaSuccess) for (auto& d : ctx->devs) if (d->device == cur) dv = d.get(); }
    LaneLock lk(dv);
    Lane* ln = lk.ln;
    CK(cudaSetDevice(dv->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // a lane is one workspace: a call on another stream waits (on the device) for the lane's previous device-path call;
    // consecutive calls take different lanes when the context has several (n_workspaces) and then overlap
    if (ln->ws_pending) CK(cudaStreamWaitEvent(s, ln->ev_ws, 0));
    const bool profiling = ctx->profiling.load();
    ProfEvents* prof = profiling ? &ln->prof : nullptr;
    if (prof) { std::memset(prof->launched, 0, sizeof prof->launched); cudaEventRecord(prof->total[0], s); cudaEventRecord(prof->h2d[0], s); cudaEventRecord(prof->h2d[1], s); }
    BatchView b{d_bytes, d_offsets, d_vocab_ids, n_prompts, total_bytes};
    enqueue_encode(b, dv->vs, dv->uc, ln->ws, d_out_ids, out_cap, d_out_offsets, d_out_counts,
                   static_cast<uint32_t>(dv->sm_count * 4), s, prof ? s : ln->aux_stream, prof ? s : ln->aux2_stream,
                   ln->ev_fork, ln->ev_join, ln->ev_join2, prof);   // profiling: one stream, so that the per-kernel times do not overlap
    CK(cudaGetLastError());
    CK(cudaEventRecord(ln->ev_ws, s));
    ln->ws_pending = true;
    ln->dev_out_cap = out_cap;
    ln->dev_want_ids = d_out_ids != nullptr;
    tl_device_lane = ln;
    if (prof) { cudaEventRecord(prof->d2h[0], s); cudaEventRecord(prof->d2h[1], s); cudaEventRecord(prof->total[1], s); }
    if (n_tokens || prof) {
        CK(cudaMemcpyAsync(ln->h_status, ln->ws.status, sizeof(DeviceStatus), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (prof) fill_profile(ln, total_bytes);
        const DeviceStatus st = *ln->h_status;
        if (n_tokens) *n_tokens = st.n_tokens;
        if (st.long_overflow || st.miss_overflow) return fail(ctx, CFBPE_EIO, "internal: long-piece list overflow");
        if (st.bad_vocab) return fail(ctx, CFBPE_ENOENT, "a prompt names a vocabulary that is not loaded");
        if (st.bad_utf8) return fail(ctx, CFBPE_EILSEQ, "a prompt holds malformed UTF-8");
        if (d_out_ids && st.n_tokens > out_cap) return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(st.n_tokens) + " ids");
    }
    return CFBPE_OK;
}

int cfbpe_encode_truncated_device(cfbpe_ctx* ctx, uint32_t n_prompts, const uint8_t* d_bytes, uint64_t total_bytes,
                                  const uint64_t* d_offsets, const uint8_t* d_vocab_ids, uint32_t max_tokens, uint32_t keep, uint32_t pad_id,
                                  const uint32_t* d_budgets, uint32_t* d_out_rows, uint32_t* d_out_kept, uint32_t* d_out_counts,
                                  uint64_t* d_out_cut, void* stream) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    tl_err.clear();
    std::shared_lock<std::shared_mutex> vocabs(ctx->vocab_mu);
    if (n_prompts > ctx->max_prompts || total_bytes > ctx->max_bytes) return fail(ctx, CFBPE_EINVAL, "batch exceeds the limits of this context");
    if (!d_offsets || !d_out_kept || (total_bytes && !d_bytes)) return fail(ctx, CFBPE_EINVAL, "device pointer is NULL");
    if (!max_tokens) return fail(ctx, CFBPE_EINVAL, "max_tokens must be at least 1");
    if (keep != CFBPE_KEEP_HEAD && keep != CFBPE_KEEP_TAIL) return fail(ctx, CFBPE_EINVAL, "keep must be CFBPE_KEEP_HEAD or CFBPE_KEEP_TAIL");
    if (!ctx->vocabs[0].loaded && !d_vocab_ids) return fail(ctx, CFBPE_ENOENT, "vocab 0 is not loaded");
    if (!ctx->loaded_mask) return fail(ctx, CFBPE_ENOENT, "no vocabulary is loaded");
    DeviceCtx* dv = ctx->devs[0].get();
    { int cur = -1; if (cudaGetDevice(&cur) == cudaSuccess) for (auto& d : ctx->devs) if (d->device == cur) dv = d.get(); }
    LaneLock lk(dv);
    Lane* ln = lk.ln;
    CK(cudaSetDevice(dv->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (ln->ws_pending) CK(cudaStreamWaitEvent(s, ln->ev_ws, 0));
    const bool profiling = ctx->profiling.load();
    ProfEvents* prof = profiling ? &ln->prof : nullptr;
    if (prof) { std::memset(prof->launched, 0, sizeof prof->launched); cudaEventRecord(prof->total[0], s); cudaEventRecord(prof->h2d[0], s); cudaEventRecord(prof->h2d[1], s); }
    // the token offsets and counts the window reads go to the lane's own buffers; the caller's counts are a copy of them
    BatchView b{d_bytes, d_offsets, d_vocab_ids, n_prompts, total_bytes};
    enqueue_encode(b, dv->vs, dv->uc, ln->ws, nullptr, 0, ln->d_out_offsets, ln->d_out_counts,
                   static_cast<uint32_t>(dv->sm_count * 4), s, prof ? s : ln->aux_stream, prof ? s : ln->aux2_stream,
                   ln->ev_fork, ln->ev_join, ln->ev_join2, prof);
    const WindowView win{max_tokens, keep, pad_id, d_budgets, d_out_rows, d_out_kept, d_out_counts, d_out_cut};
    enqueue_window(b, dv->vs, ln->ws, ln->d_out_offsets, ln->d_out_counts, win, s, prof);
    if (prof) prof->window_launches = (d_out_rows && total_bytes) ? 2 : 1;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ln->ev_ws, s));
    ln->ws_pending = true;
    ln->dev_out_cap = 0;
    ln->dev_want_ids = false;
    tl_device_lane = ln;
    if (prof) {
        cudaEventRecord(prof->d2h[0], s); cudaEventRecord(prof->d2h[1], s); cudaEventRecord(prof->total[1], s);
        CK(cudaMemcpyAsync(ln->h_status, ln->ws.status, sizeof(DeviceStatus), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        fill_profile(ln, total_bytes);
    }
    return CFBPE_OK;
}

int cfbpe_device_status(cfbpe_ctx* ctx, void* stream) {
    DeviceGuard restore_device;
    if (!ctx) return CFBPE_EINVAL;
    Lane* ln = tl_device_lane;      // the lane of this thread's last device-path call
    if (!ln) return CFBPE_OK;
    std::lock_guard<std::mutex> lock(ln->mu);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CK(cudaSetDevice(ln->device));
    CK(cudaMemcpyAsync(ln->h_status, ln->ws.status, sizeof(DeviceStatus), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (ln->h_status->long_overflow || ln->h_status->miss_overflow) return fail(ctx, CFBPE_EIO, "internal: long-piece list overflow");
    if (ln->h_status->bad_vocab) return fail(ctx, CFBPE_ENOENT, "a prompt names a vocabulary that is not loaded");
    if (ln->h_status->bad_utf8) return fail(ctx, CFBPE_EILSEQ, "a prompt holds malformed UTF-8");
    if (ln->dev_want_ids && ln->h_status->n_tokens > ln->dev_out_cap)
        return fail(ctx, CFBPE_ENOSPC, "out_cap too small: need " + std::to_string(ln->h_status->n_tokens) + " ids");
    return CFBPE_OK;
}

void* cfbpe_host_alloc(cfbpe_ctx* ctx, size_t size) {
    DeviceGuard restore_device;
    if (!ctx) return nullptr;
    void* p = nullptr;
    cudaSetDevice(ctx->devs[0]->device);
    if (cudaMallocHost(&p, size ? size : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void cfbpe_host_free(cfbpe_ctx* ctx, void* ptr) {
    DeviceGuard restore_device;
    if (!ctx || !ptr) return;
    cudaFreeHost(ptr);
}

int cfbpe_profile_enable(cfbpe_ctx* ctx, int on) {
    if (!ctx) return CFBPE_EINVAL;
    ctx->profiling.store(on != 0);
    tl_profile_ready = false;
    return CFBPE_OK;
}
int cfbpe_profile_read(cfbpe_ctx* ctx, cfbpe_profile* out) {
    DeviceGuard restore_device;
    if (!ctx || !out) return CFBPE_EINVAL;
    if (!tl_profile_ready) return CFBPE_ENOENT;
    *out = tl_profile;
    return CFBPE_OK;
}

}  // extern "C"
