/*
 * cfbpe.h -- C ABI of the B200-native batched BPE tokenizer (libcfbpe.so).
 *
 * This is the drop-in boundary for cyberfabric-core's LLM Gateway tokenizer /
 * usage-meter worker.  The reference tree has no tokenizer code to replace
 * (modules/llm-gateway/README.md:51-52 lists the implementation crate and plugins as
 * "planned"; SURVEY.md F1), so each entry point cites the *spec'd consumer* it serves and
 * the ModKit convention it follows instead of a replaced function:
 *
 *   cfbpe_create / cfbpe_destroy   plugin Module::init / stop: one-time device context,
 *                                  tables and staging buffers, created where a ModKit plugin
 *                                  registers its scoped client
 *                                  (modules/system/tenant-resolver/plugins/static-tr-plugin/src/module.rs:43-88).
 *   cfbpe_vocab_load / _export / _import
 *                                  the model-registry vocab loader that does not exist yet:
 *                                  `Model` has no tokenizer field
 *                                  (modules/model-registry/docs/PRD.md:196-209); rank-file format
 *                                  per tiktoken/load.py:160-172.  export/import move the packed
 *                                  device tables so one rank parses and the host layer broadcasts
 *                                  them (NCCL) to the other GPUs of the box.
 *   cfbpe_encode_batch             `TokenizerPluginClient::encode_batch` (llm-gateway::tokenizer):
 *                                  token ids for a packed multi-tenant prompt buffer.
 *   cfbpe_count_batch              `llm-gateway::usage::count_tokens`: feeds
 *                                  Usage.input_tokens (modules/llm-gateway/llm-gateway-sdk/schemas/core/usage.v1.schema.json:8-12)
 *                                  and check_budget / report_usage (modules/llm-gateway/docs/DESIGN.md:833-855).
 *   cfbpe_encode_batch_device      same path with inputs/outputs already resident in HBM
 *                                  (for callers that keep token ids on the GPU).
 *   cfbpe_encode_truncated[_device] a prompt cut to a token budget: the request may not exceed the provider's context window
 *                                  (modules/llm-gateway/docs/DESIGN.md:102-106); fixed-length id rows and the byte cut of each prompt.
 *
 * Conventions (SURVEY.md section 8(b)): 0 = ok, negative errno-style code = error; the caller
 * owns every buffer it passes and the library never retains a caller pointer past return;
 * the library owns device memory, pinned staging and streams; nothing throws across the
 * ABI; entry points taking a ctx may be called from several host threads: a context holds
 * cfbpe_config.n_workspaces independent call lanes per device (calls wait only when all are
 * busy; vocabulary loads exclude running calls), the last error is kept per thread, and every
 * entry point leaves the caller's current CUDA device as it found it.  There is NO CPU fallback: cfbpe_create fails with
 * CFBPE_ENODEV when no sm_100 device is present.
 *
 * Results are bit-exact with tiktoken 0.12.0 CoreBPE.encode_ordinary for the same rank
 * file and pattern (see oracle/ and tests/).
 */
#ifndef CFBPE_H
#define CFBPE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CFBPE_API __attribute__((visibility("default")))
#else
#define CFBPE_API
#endif

#define CFBPE_ABI_VERSION 1u

/* error codes (negative errno values) */
#define CFBPE_OK 0
#define CFBPE_ENOENT (-2)    /* unknown vocab id */
#define CFBPE_EIO (-5)       /* CUDA runtime failure; see cfbpe_last_error */
#define CFBPE_ENOMEM (-12)
#define CFBPE_ENODEV (-19)   /* no usable sm_100 device */
#define CFBPE_EINVAL (-22)   /* bad argument: null pointer, non-monotonic offsets, oversize batch, bad rank file */
#define CFBPE_ENOSPC (-28)   /* out_cap too small; required id count is in out_offsets[n_prompts] */
#define CFBPE_EILSEQ (-84)   /* a prompt holds malformed UTF-8 (tiktoken only accepts valid text) */

/* rank-file formats */
#define CFBPE_FORMAT_TIKTOKEN 0u     /* "<base64 token> <rank>\n" lines */
#define CFBPE_FORMAT_TEKKEN_JSON 1u  /* mistral_common tekken_*.json */

/* pre-tokenizer patterns */
#define CFBPE_PATTERN_CL100K 0u
#define CFBPE_PATTERN_O200K 1u
#define CFBPE_PATTERN_LLAMA3 2u
#define CFBPE_PATTERN_TEKKEN 3u
#define CFBPE_PATTERN_COUNT 4u

#define CFBPE_MAX_VOCABS 8u

typedef struct cfbpe_ctx cfbpe_ctx; /* opaque */

#define CFBPE_MAX_DEVICES 8

typedef struct cfbpe_config {
    uint32_t struct_size;     /* sizeof(cfbpe_config), for forward compatibility: a caller built against the five-field struct of
                                 ABI version 1 (24 bytes) still works, and gets one device and one workspace */
    int32_t device;           /* CUDA device ordinal (used when n_devices == 0) */
    uint64_t max_batch_bytes; /* largest packed prompt buffer one DEVICE takes in one call (0 = 256 MiB) */
    uint32_t max_prompts;     /* largest n_prompts of one call (0 = 1 Mi); each workspace holds 16 bytes of device memory per prompt
                                 for the budgets, kept counts and cuts of cfbpe_encode_truncated */
    uint32_t flags;           /* reserved, 0 */
    /* SURVEY.md section 8(b): cfbpe_create(cfg: devices[], n_devices, ...) */
    int32_t devices[CFBPE_MAX_DEVICES]; /* CUDA ordinals of a multi-device context */
    uint32_t n_devices;       /* 0 = single device (`device`); > 1: the packed tables are broadcast with NCCL (libnccl.so.2 is
                                 dlopen'ed; without it cfbpe_create fails with CFBPE_EIO) and a host batch is spread over the
                                 devices -- its sub-batches round-robin, token ranks chained over NVLink peer memory, when
                                 every device can hold the whole batch (<= max_batch_bytes); else one contiguous shard of
                                 whole prompts a device, the shard totals gathered with NCCL */
    uint32_t n_workspaces;    /* independent workspaces per device (0 = 1, at most 16): that many calls run concurrently on the
                                 context; each costs ~33 bytes of device memory per byte of max_batch_bytes */
} cfbpe_config;

typedef struct cfbpe_vocab_info {
    uint32_t n_ranks;
    uint32_t pattern_id;
    uint32_t max_token_len;
    uint32_t n_pair_entries;  /* (left,right)->merged entries in the all-splits pair table */
    uint64_t table_bytes;     /* size of the packed device tables (= export size) */
} cfbpe_vocab_info;

/* per-call device timings, filled when profiling is on (cfbpe_profile_enable) */
#define CFBPE_NUM_KERNELS 10
typedef struct cfbpe_profile {
    float kernel_ms[CFBPE_NUM_KERNELS]; /* 0 pretok_split, 1 bpe_encode, 2 bpe_long, 3 flag_count, 4 tile_scan, 5 emit_compact (+ offsets), 6 bpe_list, 7 long_scan, 8 bpe_merge,
                                           9 window (cfbpe_encode_truncated only: window_select + emit_window; 0 otherwise) */
    uint32_t kernel_launches[CFBPE_NUM_KERNELS];
    float h2d_ms, d2h_ms, total_ms;
    uint64_t n_tokens, n_bytes, n_long_pieces;
    uint64_t n_long_bytes, n_long_tokens; /* bytes in / ids out of the long-piece kernels */
    uint64_t n_miss_pieces;               /* short pieces that were not one token (merged by bpe_merge) */
    uint64_t n_list_pieces, n_list_parts; /* big pieces whose list phase ran in bpe_list, and their parts when it began */
    uint64_t n_extra_tokens;              /* tokens of the merged short pieces (the dense `extras` list of bpe_merge) */
} cfbpe_profile;

CFBPE_API int cfbpe_abi_version(void);
/* sha256 (hex, first 16 chars) of the sources this binary was built from; lets the host layer refuse a stale build */
CFBPE_API const char *cfbpe_build_id(void);

CFBPE_API int cfbpe_create(const cfbpe_config *cfg, cfbpe_ctx **out);
CFBPE_API void cfbpe_destroy(cfbpe_ctx *ctx);
/* NUL-terminated description of the last failure of the CALLING THREAD (valid until its next call): entry points run
 * concurrently on one context, so the message is kept per thread, not per context */
CFBPE_API const char *cfbpe_last_error(const cfbpe_ctx *ctx);

/* Parse a rank file, build the lookup tables on the host and upload them.
 * max_ranks: keep only ranks < max_ranks (0 = all). */
CFBPE_API int cfbpe_vocab_load(cfbpe_ctx *ctx, uint32_t vocab_id, const uint8_t *ranks_file, size_t len,
                     uint32_t format, uint32_t pattern_id, uint32_t max_ranks);
CFBPE_API int cfbpe_vocab_get_info(const cfbpe_ctx *ctx, uint32_t vocab_id, cfbpe_vocab_info *out);
/* Copy the packed tables out (size query: buf = NULL, cap = 0) / install packed tables
 * produced by cfbpe_vocab_export on another rank. */
CFBPE_API int cfbpe_vocab_export(const cfbpe_ctx *ctx, uint32_t vocab_id, uint8_t *buf, uint64_t cap, uint64_t *size);
CFBPE_API int cfbpe_vocab_import(cfbpe_ctx *ctx, uint32_t vocab_id, const uint8_t *buf, uint64_t size);

/* Encode n_prompts prompts.  bytes/offsets: packed UTF-8, prompt i = bytes[offsets[i] .. offsets[i+1]),
 * offsets[0] must be 0.  vocab_ids: per-prompt vocab id or NULL (all vocab 0).
 * out_ids: room for out_cap ids; out_offsets: n_prompts+1; out_counts: n_prompts (may be NULL).
 * Host pointers; pinned buffers from cfbpe_host_alloc are DMA'd directly, others are staged. */
CFBPE_API int cfbpe_encode_batch(cfbpe_ctx *ctx, uint32_t n_prompts, const uint8_t *bytes, const uint64_t *offsets,
                       const uint8_t *vocab_ids, uint32_t *out_ids, uint64_t out_cap, uint64_t *out_offsets,
                       uint32_t *out_counts);
/* Token counts only (no id stream leaves the device). */
CFBPE_API int cfbpe_count_batch(cfbpe_ctx *ctx, uint32_t n_prompts, const uint8_t *bytes, const uint64_t *offsets,
                      const uint8_t *vocab_ids, uint32_t *out_counts);

/* Truncated encode: every prompt cut to a token budget, as fixed-length rows of ids.
 * Prompt i has c_i tokens (its full encode_ordinary) and keeps k_i = min(c_i, budgets[i], max_tokens) of them (budgets may be
 * NULL: max_tokens for every prompt; max_tokens >= 1).
 *   keep = CFBPE_KEEP_HEAD: ids[0 : k_i]; out_cut[i] = the byte offset inside the prompt where token k_i starts, or the prompt's
 *          length when nothing was dropped; the kept tokens cover exactly prompt[0 : cut].
 *   keep = CFBPE_KEEP_TAIL: ids[c_i - k_i : c_i]; out_cut[i] = where the first kept token starts, or 0 when nothing was dropped;
 *          the kept tokens cover exactly prompt[cut : len].
 * out_rows (may be NULL: no id leaves the device) is n_prompts x max_tokens uint32, row-major: row i holds the k_i kept ids
 * left-aligned, then pad_id up to max_tokens.  out_kept[i] = k_i (required), out_counts[i] = c_i (may be NULL), out_cut[i]
 * (may be NULL).
 * The kept ids are a slice of the full encoding.  Re-encoding the kept bytes need not give the same ids: the pre-tokenizer's
 * lookahead (\s+(?!\S)) sees different text at the cut.  And a cut may fall inside a multi-byte UTF-8 character (byte-level tokens
 * split CJK characters and emoji): out_cut is the token boundary exactly as it is, never moved to a character boundary.
 * Errors as cfbpe_encode_batch (EILSEQ, ENOENT, EINVAL for bad offsets and limits), and CFBPE_EINVAL for max_tokens == 0, an
 * unknown keep, a NULL out_kept, or, with out_rows, n_prompts x max_tokens > max_batch_bytes (the rows are staged in the
 * context's id buffer).  Never CFBPE_ENOSPC: the caller sizes the rows. */
#define CFBPE_KEEP_HEAD 0u
#define CFBPE_KEEP_TAIL 1u
CFBPE_API int cfbpe_encode_truncated(cfbpe_ctx *ctx, uint32_t n_prompts, const uint8_t *bytes, const uint64_t *offsets,
                                     const uint8_t *vocab_ids, uint32_t max_tokens, uint32_t keep, uint32_t pad_id,
                                     const uint32_t *budgets, uint32_t *out_rows, uint32_t *out_kept, uint32_t *out_counts,
                                     uint64_t *out_cut);

/* Decode (SURVEY.md section 8(f) item 2; tiktoken CoreBPE.decode_bytes): out_bytes = the concatenation of the tokens' bytes.
 * ids: the packed token ids of n_seqs sequences, id_offsets[n_seqs + 1] their boundaries (in ids), vocab_ids[n_seqs] or NULL.
 * out_offsets[n_seqs + 1]: byte boundaries of the decoded sequences in out_bytes.  CFBPE_ENOSPC if out_cap is too small
 * (out_offsets[n_seqs] = bytes needed), CFBPE_EINVAL for an id outside its vocabulary or a batch beyond the context's limits
 * (at most max_batch_bytes ids and max_batch_bytes decoded bytes).  Host buffers; no reference interface exists for it
 * (the reference ships no tokenizer: SURVEY.md F1). */
CFBPE_API int cfbpe_decode_batch(cfbpe_ctx* ctx, uint32_t n_seqs, const uint32_t* ids, const uint64_t* id_offsets,
                                 const uint8_t* vocab_ids, uint8_t* out_bytes, uint64_t out_cap, uint64_t* out_offsets);

/* Same path on device-resident buffers, enqueued on `stream` (a cudaStream_t; NULL = the legacy
 * default stream).  d_bytes must be readable for 32 bytes past total_bytes (the kernels read whole 16-byte
 * groups); the contents of that padding do not matter.  d_out_ids may be NULL (count only).  n_tokens (host, may be NULL) is written
 * after an internal stream sync; with n_tokens == NULL the call is fully asynchronous and
 * d_out_offsets[n_prompts] holds the total.  Malformed UTF-8 is reported by the next call that
 * synchronises (or cfbpe_device_status). */
CFBPE_API int cfbpe_encode_batch_device(cfbpe_ctx *ctx, uint32_t n_prompts, const uint8_t *d_bytes, uint64_t total_bytes,
                              const uint64_t *d_offsets, const uint8_t *d_vocab_ids, uint32_t *d_out_ids,
                              uint64_t out_cap, uint64_t *d_out_offsets, uint32_t *d_out_counts,
                              uint64_t *n_tokens, void *stream);
/* cfbpe_encode_truncated on device-resident buffers, asynchronous as cfbpe_encode_batch_device (d_bytes padded by 32 readable
 * bytes; errors through cfbpe_device_status).  d_budgets, d_out_rows, d_out_counts, d_out_cut may be NULL; no limit on
 * n_prompts x max_tokens (the rows are the caller's buffer).  The context's own offset and count buffers hold the token offsets
 * the window reads. */
CFBPE_API int cfbpe_encode_truncated_device(cfbpe_ctx *ctx, uint32_t n_prompts, const uint8_t *d_bytes, uint64_t total_bytes,
                                            const uint64_t *d_offsets, const uint8_t *d_vocab_ids, uint32_t max_tokens,
                                            uint32_t keep, uint32_t pad_id, const uint32_t *d_budgets, uint32_t *d_out_rows,
                                            uint32_t *d_out_kept, uint32_t *d_out_counts, uint64_t *d_out_cut, void *stream);
/* Synchronise `stream` and return the status word of the last device call (0, CFBPE_EILSEQ, CFBPE_ENOSPC). */
CFBPE_API int cfbpe_device_status(cfbpe_ctx *ctx, void *stream);

/* page-locked host memory the DMA engines can read without a staging copy */
CFBPE_API void *cfbpe_host_alloc(cfbpe_ctx *ctx, size_t size);
CFBPE_API void cfbpe_host_free(cfbpe_ctx *ctx, void *ptr);

/* CUDA-event timing of each kernel of the following calls (adds event records, no syncs) */
CFBPE_API int cfbpe_profile_enable(cfbpe_ctx *ctx, int on);
CFBPE_API int cfbpe_profile_read(cfbpe_ctx *ctx, cfbpe_profile *out);

#ifdef __cplusplus
}
#endif
#endif /* CFBPE_H */
