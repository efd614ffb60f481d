//! The plugin's service: owns the device context, resolves vocabularies, maps errors, keeps CUDA syncs off the runtime.

use std::collections::HashMap;
use std::sync::Arc;

use async_trait::async_trait;
use cfbpe_sys::{Ctx, NativeError, CFBPE_KEEP_HEAD, CFBPE_KEEP_TAIL};
use llm_gateway_sdk::{
    CountTokensRequest, DecodeBatchRequest, DecodeBatchResponse, EncodeBatchRequest, EncodeBatchResponse, Keep, TokenizerError,
    TokenizerPluginClient, TruncateBatchRequest, TruncateBatchResponse, VocabRef,
};
use modkit_security::SecurityContext;
use sha2::{Digest, Sha256};

use crate::batcher::CountBatcher;
use crate::config::{GpuBpeTokenizerPluginConfig, Pattern, RankFileFormat};

pub struct Service {
    native: Arc<Ctx>,
    /// vocabulary name or canonical model id -> slot on the device context
    slots: HashMap<String, u8>,
    names: Vec<String>,
    batcher: CountBatcher,
}

fn map_native(e: NativeError) -> TokenizerError {
    match e.code {
        cfbpe_sys::CFBPE_EINVAL | cfbpe_sys::CFBPE_EILSEQ | cfbpe_sys::CFBPE_ENOSPC => TokenizerError::InvalidInput(e.message),
        cfbpe_sys::CFBPE_ENOENT => TokenizerError::VocabNotFound { vocab: e.message },
        cfbpe_sys::CFBPE_ENODEV | cfbpe_sys::CFBPE_ENOMEM => TokenizerError::ServiceUnavailable(e.message),
        _ => TokenizerError::Internal(e.message),
    }
}

impl Service {
    /// Blocking: called from `spawn_blocking` in `Module::init`.
    pub fn from_config(cfg: &GpuBpeTokenizerPluginConfig) -> anyhow::Result<Self> {
        let native = Ctx::create(&cfg.devices, cfg.max_batch_bytes, cfg.max_prompts, cfg.workspaces)
            .map_err(|e| anyhow::anyhow!("no B200 device context (there is no CPU fallback): {e}"))?;
        let mut slots = HashMap::new();
        let mut names = Vec::new();
        for (slot, v) in cfg.vocabs.iter().enumerate() {
            anyhow::ensure!(slot < cfbpe_sys::CFBPE_MAX_VOCABS as usize, "at most {} vocabularies per context", cfbpe_sys::CFBPE_MAX_VOCABS);
            let file = std::fs::read(&v.path)?;
            let sha = format!("{:x}", Sha256::digest(&file));
            anyhow::ensure!(sha.eq_ignore_ascii_case(&v.sha256), "{}: sha256 {sha} does not match the configured {}", v.path, v.sha256);
            let format = match v.format {
                RankFileFormat::Tiktoken => cfbpe_sys::CFBPE_FORMAT_TIKTOKEN,
                RankFileFormat::TekkenJson => cfbpe_sys::CFBPE_FORMAT_TEKKEN_JSON,
            };
            let pattern = match v.pattern {
                Pattern::Cl100k => 0,
                Pattern::O200k => 1,
                Pattern::Llama3 => 2,
                Pattern::Tekken => 3,
            };
            native.vocab_load(slot as u32, &file, format, pattern, v.max_ranks).map_err(|e| anyhow::anyhow!("{}: {e}", v.name))?;
            slots.insert(v.name.clone(), slot as u8);
            for m in &v.models {
                slots.insert(m.clone(), slot as u8);
            }
            names.push(v.name.clone());
        }
        let native = Arc::new(native);
        let batcher = CountBatcher::start(native.clone(), cfg.batch_bytes.min(cfg.max_batch_bytes), cfg.max_prompts, cfg.batch_wait_us);
        Ok(Self { native, slots, names, batcher })
    }

    pub fn vocab_names(&self) -> &[String] {
        &self.names
    }

    fn slot(&self, v: &VocabRef) -> Result<u8, TokenizerError> {
        self.slots.get(&v.0).copied().ok_or_else(|| TokenizerError::VocabNotFound { vocab: v.0.clone() })
    }

    /// one vocabulary id per prompt, or `None` when the whole batch uses slot 0
    fn vocab_ids(&self, vocab: &VocabRef, per_prompt: Option<&[VocabRef]>, index: Option<&[u8]>, n: usize) -> Result<Option<Vec<u8>>, TokenizerError> {
        if let (Some(table), Some(idx)) = (per_prompt, index) {
            // a table of distinct vocabularies + one index per prompt
            if idx.len() != n {
                return Err(TokenizerError::InvalidInput("vocab_index must hold one entry per prompt".to_owned()));
            }
            let lut = table.iter().map(|r| self.slot(r)).collect::<Result<Vec<_>, _>>()?;
            return idx
                .iter()
                .map(|&i| lut.get(i as usize).copied().ok_or_else(|| TokenizerError::InvalidInput(format!("vocab_index names entry {i} of {} vocabularies", lut.len()))))
                .collect::<Result<Vec<_>, _>>()
                .map(Some);
        }
        match per_prompt {
            Some(v) if v.len() != n => Err(TokenizerError::InvalidInput("vocabs_per_prompt must name one vocabulary per prompt".to_owned())),
            Some(v) => v.iter().map(|r| self.slot(r)).collect::<Result<Vec<_>, _>>().map(Some),
            None => {
                let s = self.slot(vocab)?;
                Ok(if s == 0 { None } else { Some(vec![s; n.max(1)]) })
            }
        }
    }
}

#[async_trait]
impl TokenizerPluginClient for Service {
    async fn encode_batch(&self, _ctx: &SecurityContext, req: EncodeBatchRequest) -> Result<EncodeBatchResponse, TokenizerError> {
        let n = req.offsets.len().saturating_sub(1);
        let vid = self.vocab_ids(&req.vocab, req.vocabs_per_prompt.as_deref(), req.vocab_index.as_deref(), n)?;
        let native = self.native.clone();
        // never block a tokio worker on a CUDA synchronisation (precedent: modules/file-parser/src/infra/parsers/html_parser.rs:47)
        let out = tokio::task::spawn_blocking(move || native.encode_batch(&req.bytes, &req.offsets, vid.as_deref()))
            .await
            .map_err(|e| TokenizerError::Internal(e.to_string()))?
            .map_err(map_native)?;
        Ok(EncodeBatchResponse { ids: out.ids, offsets: out.offsets, counts: out.counts })
    }

    async fn count_tokens(&self, _ctx: &SecurityContext, req: CountTokensRequest) -> Result<Vec<u32>, TokenizerError> {
        let n = req.offsets.len().saturating_sub(1);
        let vid = self.vocab_ids(&req.vocab, req.vocabs_per_prompt.as_deref(), req.vocab_index.as_deref(), n)?;
        // small requests (a chat message is a few KB) ride in a shared device batch; large ones go straight through
        if (req.bytes.len() as u64) < self.batcher.direct_threshold() {
            return self.batcher.count(req.bytes, req.offsets, vid).await;
        }
        let native = self.native.clone();
        tokio::task::spawn_blocking(move || native.count_batch(&req.bytes, &req.offsets, vid.as_deref()))
            .await
            .map_err(|e| TokenizerError::Internal(e.to_string()))?
            .map_err(map_native)
    }

    async fn decode_batch(&self, _ctx: &SecurityContext, req: DecodeBatchRequest) -> Result<DecodeBatchResponse, TokenizerError> {
        let n = req.offsets.len().saturating_sub(1);
        let vid = self.vocab_ids(&req.vocab, req.vocabs_per_prompt.as_deref(), req.vocab_index.as_deref(), n)?;
        let native = self.native.clone();
        let (bytes, offsets) = tokio::task::spawn_blocking(move || native.decode_batch(&req.ids, &req.offsets, vid.as_deref()))
            .await
            .map_err(|e| TokenizerError::Internal(e.to_string()))?
            .map_err(map_native)?;
        Ok(DecodeBatchResponse { bytes, offsets })
    }

    async fn truncate_batch(&self, _ctx: &SecurityContext, req: TruncateBatchRequest) -> Result<TruncateBatchResponse, TokenizerError> {
        let n = req.offsets.len().saturating_sub(1);
        let vid = self.vocab_ids(&req.vocab, req.vocabs_per_prompt.as_deref(), req.vocab_index.as_deref(), n)?;
        let keep = match req.keep { Keep::Head => CFBPE_KEEP_HEAD, Keep::Tail => CFBPE_KEEP_TAIL };
        let native = self.native.clone();
        let out = tokio::task::spawn_blocking(move || {
            native.encode_truncated(&req.bytes, &req.offsets, vid.as_deref(), req.max_tokens, keep, req.pad_id, req.budgets.as_deref(), req.want_ids)
        })
        .await
        .map_err(|e| TokenizerError::Internal(e.to_string()))?
        .map_err(map_native)?;
        Ok(TruncateBatchResponse { rows: out.rows, kept: out.kept, counts: out.counts, cut: out.cut })
    }
}

pub(crate) fn map_native_error(e: NativeError) -> TokenizerError {
    map_native(e)
}
