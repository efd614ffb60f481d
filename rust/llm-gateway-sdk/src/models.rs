//! Request / response models of the tokenizer API.
//!
//! A batch is ONE packed buffer: the UTF-8 bytes of all prompts back to back plus `n + 1` byte offsets — the layout the device
//! path reads with coalesced 16-byte loads; requests of many tenants share a batch, each prompt naming its vocabulary.

use std::collections::BTreeMap;

use bytes::Bytes;
use serde::{Deserialize, Serialize};

/// Names a vocabulary: a registry name (`cl100k_base`) or a model-registry canonical id (`openai::gpt-4`,
/// `{provider_slug}::{provider_model_id}`, `modules/model-registry/docs/PRD.md:197`).
#[derive(Debug, Clone, PartialEq, Eq, Hash, Serialize, Deserialize)]
pub struct VocabRef(pub String);

#[derive(Debug, Clone)]
pub struct EncodeBatchRequest {
    pub vocab: VocabRef,
    /// packed UTF-8 of all prompts
    pub bytes: Bytes,
    /// `n + 1` offsets into `bytes`, `offsets[0] == 0`, non-decreasing
    pub offsets: Vec<u64>,
    /// multi-tenant batches: one vocabulary per prompt (overrides `vocab`)
    pub vocabs_per_prompt: Option<Vec<VocabRef>>,
    /// with it, `vocabs_per_prompt` lists the DISTINCT vocabularies and `vocab_index[i]` picks prompt i's
    /// (a 65 536-prompt batch carries three names and 64 KiB of indices, not 65 536 strings)
    pub vocab_index: Option<Vec<u8>>,
}

#[derive(Debug, Clone, Default)]
pub struct EncodeBatchResponse {
    /// dense id stream of all prompts (tiktoken `encode_ordinary` semantics, bit-exact)
    pub ids: Vec<u32>,
    /// `n + 1` offsets into `ids`
    pub offsets: Vec<u64>,
    pub counts: Vec<u32>,
}

#[derive(Debug, Clone)]
pub struct CountTokensRequest {
    pub vocab: VocabRef,
    pub bytes: Bytes,
    pub offsets: Vec<u64>,
    pub vocabs_per_prompt: Option<Vec<VocabRef>>,
    pub vocab_index: Option<Vec<u8>>,
}

/// Which end of a prompt a truncation keeps.
#[derive(Debug, Clone, Copy, PartialEq, Eq, Default, Serialize, Deserialize)]
#[serde(rename_all = "snake_case")]
pub enum Keep {
    #[default]
    Head,
    Tail,
}

/// Every prompt cut to `k_i = min(count_i, budgets[i], max_tokens)` tokens: the first `k_i` (`Keep::Head`) or the last (`Keep::Tail`)
/// of its full encoding.  The kept ids are a slice of that encoding (re-encoding the kept bytes need not give the same ids), and the
/// cut is the token boundary as it is, possibly inside a multi-byte UTF-8 character.
#[derive(Debug, Clone)]
pub struct TruncateBatchRequest {
    pub vocab: VocabRef,
    pub bytes: Bytes,
    pub offsets: Vec<u64>,
    /// ids per row, >= 1
    pub max_tokens: u32,
    pub keep: Keep,
    pub pad_id: u32,
    /// one budget per prompt, or `max_tokens` for every prompt
    pub budgets: Option<Vec<u32>>,
    /// false: kept counts and cuts only, no id leaves the device
    pub want_ids: bool,
    pub vocabs_per_prompt: Option<Vec<VocabRef>>,
    pub vocab_index: Option<Vec<u8>>,
}

#[derive(Debug, Clone, Default)]
pub struct TruncateBatchResponse {
    /// `n x max_tokens`, row-major: prompt i's kept ids left-aligned, then `pad_id` (empty when `want_ids` is false)
    pub rows: Vec<u32>,
    pub kept: Vec<u32>,
    /// the untruncated counts
    pub counts: Vec<u32>,
    /// byte offset of the cut inside prompt i: `Head` keeps `prompt[..cut]`, `Tail` keeps `prompt[cut..]`
    pub cut: Vec<u64>,
}

#[derive(Debug, Clone)]
pub struct DecodeBatchRequest {
    pub vocab: VocabRef,
    pub ids: Vec<u32>,
    pub offsets: Vec<u64>,
    pub vocabs_per_prompt: Option<Vec<VocabRef>>,
    pub vocab_index: Option<Vec<u8>>,
}

#[derive(Debug, Clone, Default)]
pub struct DecodeBatchResponse {
    /// the sequences' bytes back to back (tiktoken `decode_bytes`: not necessarily valid UTF-8)
    pub bytes: Vec<u8>,
    pub offsets: Vec<u64>,
}

/// Special tokens of a vocabulary and which of them a request may spell out (tiktoken `Encoding.encode`: by default none is
/// allowed and every one is disallowed, so user text that spells a control token is refused, not turned into one).
#[derive(Debug, Clone, Default)]
pub struct SpecialTokens {
    pub ids: BTreeMap<String, u32>,
    pub allowed: Vec<String>,
    pub disallow_all_others: bool,
}

/// How a provider frames a list of chat messages into the token stream it bills as `Usage.input_tokens`
/// (Python mirror: `cfbpe/plugin.py:ChatTemplate`).  Message content is always ordinary text: a message that spells a control
/// token costs the pieces of that spelling and never becomes the control token.
#[derive(Debug, Clone, PartialEq, Eq)]
pub enum ChatTemplate {
    /// a fixed number of framing tokens a message (OpenAI ChatML accounting: 3 a message, 1 a name, 3 to prime the reply)
    Overhead { tokens_per_message: u32, tokens_per_name: u32, reply_priming: u32 },
    /// the conversation rendered to text around control tokens (Llama 3, Mistral): `bos`, then per message
    /// `message_prefix` (with `{role}`) + content + `message_suffix`, then `generation_prompt`; every string of
    /// `special_tokens` counts one token, the text between two of them is tokenised as ONE stretch of ordinary text
    Rendered { bos: String, message_prefix: String, message_suffix: String, generation_prompt: String, special_tokens: Vec<String> },
}

/// `gts.x.llmgw.core.usage.v1~` (`llm-gateway-sdk/schemas/core/usage.v1.schema.json:8-12`)
#[derive(Debug, Clone, Copy, Default, PartialEq, Eq, Serialize, Deserialize)]
pub struct Usage {
    pub input_tokens: u64,
    pub output_tokens: u64,
}
