//! LLM Gateway SDK — tokenizer part.
//!
//! - [`TokenizerClient`]: public API for consumers (`hub.get::<dyn TokenizerClient>()`), e.g. the chat engine's budget check
//!   (`modules/llm-gateway/docs/DESIGN.md:833-855`)
//! - [`TokenizerPluginClient`]: plugin API (scoped in `ClientHub` by GTS instance id); the name ends in `PluginClient` (lint DE0503)
//! - [`EncodeBatchRequest`] …: models;  [`TokenizerError`]: errors;  [`TokenizerPluginSpecV1`]: GTS schema for plugin discovery
//!
//! Layout follows `modules/system/tenant-resolver/tenant-resolver-sdk/src/lib.rs`.  NOT COMPILED where this file lives (no Rust
//! toolchain); the same names, argument meaning and error behaviour are implemented and tested in
//! `cyberfabric-core_b200/cfbpe/plugin.py`.

pub mod api;
pub mod error;
pub mod gts;
pub mod models;
pub mod plugin_api;

pub use api::TokenizerClient;
pub use error::TokenizerError;
pub use gts::TokenizerPluginSpecV1;
pub use models::{
    ChatTemplate, CountTokensRequest, DecodeBatchRequest, DecodeBatchResponse, EncodeBatchRequest, EncodeBatchResponse, Keep, SpecialTokens, TruncateBatchRequest, TruncateBatchResponse, Usage, VocabRef,
};
pub use plugin_api::TokenizerPluginClient;
