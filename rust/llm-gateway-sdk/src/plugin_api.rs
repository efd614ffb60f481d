//! Plugin API trait of tokenizer implementations (shape of `tenant-resolver-sdk/src/plugin_api.rs:28-47`).

use async_trait::async_trait;
use modkit_security::SecurityContext;

use crate::error::TokenizerError;
use crate::models::{
    CountTokensRequest, DecodeBatchRequest, DecodeBatchResponse, EncodeBatchRequest, EncodeBatchResponse, TruncateBatchRequest,
    TruncateBatchResponse,
};

/// Each plugin registers this trait with a scoped `ClientHub` entry using its GTS instance id as the scope.  Clients are
/// `Arc<dyn … + Send + Sync>` shared by all tokio tasks (`libs/modkit/src/client_hub.rs:142-165`): calls are concurrent and
/// re-entrant, and an implementation must not block a runtime worker on a device synchronisation (use `spawn_blocking`).
#[async_trait]
pub trait TokenizerPluginClient: Send + Sync {
    /// Token ids of every prompt of the batch.
    ///
    /// # Errors
    /// `InvalidInput` (offsets, malformed UTF-8, batch too large), `VocabNotFound`, `ServiceUnavailable`, `Internal`.
    async fn encode_batch(&self, ctx: &SecurityContext, req: EncodeBatchRequest) -> Result<EncodeBatchResponse, TokenizerError>;

    /// Token count of every prompt of the batch (`usage::count_tokens`); same errors.
    async fn count_tokens(&self, ctx: &SecurityContext, req: CountTokensRequest) -> Result<Vec<u32>, TokenizerError>;

    /// ids -> bytes; `InvalidInput` for an id outside its vocabulary.
    async fn decode_batch(&self, ctx: &SecurityContext, req: DecodeBatchRequest) -> Result<DecodeBatchResponse, TokenizerError>;

    /// Every prompt cut to a token budget: fixed-length id rows, kept and full counts, the byte cut of each prompt; the errors
    /// of `encode_batch`, and `InvalidInput` for `max_tokens == 0` or rows beyond the plugin's batch limit.
    async fn truncate_batch(&self, ctx: &SecurityContext, req: TruncateBatchRequest) -> Result<TruncateBatchResponse, TokenizerError>;
}
