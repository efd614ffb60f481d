"""Python mirror of the ModKit plugin surface the tokenizer sits behind.

The Rust toolchain is absent from this image (SURVEY.md F7), so the host side above the C ABI
is written here with the names, argument meaning and error behaviour a ModKit plugin has
(INTEGRATION.md shows the Rust crates a maintainer would add).  Conventions mirrored, with
the reference file each one follows:

* plugin trait name ends in `PluginClient` (lint DE0503, dylint_lints/README.md:36); methods
  take the SecurityContext first and return Result<_, XError>
  (modules/system/tenant-resolver/tenant-resolver-sdk/src/plugin_api.rs:28-47);
* error enum with NoPluginAvailable / ServiceUnavailable(String) / Internal(String)
  (modules/system/tenant-resolver/tenant-resolver-sdk/src/error.rs:7-34);
* a plugin registers a GTS instance {id, vendor, priority, properties}
  (libs/modkit/src/gts/plugin.rs:12-17) and a client scoped by that instance id
  (libs/modkit/src/client_hub.rs:142-234); the gateway picks vendor match, lowest priority
  (libs/modkit/src/plugins/mod.rs:136-191) and resolves lazily, once;
* token counts feed Usage.input_tokens >= 0
  (modules/llm-gateway/llm-gateway-sdk/schemas/core/usage.v1.schema.json:8-12) and are the sum over a
  request's TextContent.text parts (schemas/content/text_content.v1.schema.json,
  schemas/core/message.v1.schema.json).

Prompt text is never logged (modules/llm-gateway/docs/DESIGN.md:120-124): only sizes and counts.
"""
from __future__ import annotations

import threading
import uuid
from dataclasses import dataclass, field
from typing import Tuple, Dict, List, Optional, Sequence

import numpy as np

from . import _native as N
from . import vocabs as V


# --------------------------------------------------------------------------- errors
class TokenizerError(Exception):
    """base of the SDK error enum (`TokenizerError` in the planned llm-gateway-sdk)"""


class NoPluginAvailable(TokenizerError):
    pass


class ServiceUnavailable(TokenizerError):
    pass


class Internal(TokenizerError):
    pass


class InvalidInput(TokenizerError):
    """bad offsets / malformed UTF-8 / oversize batch (maps to RFC 9457 Problem 400)"""


class VocabNotFound(TokenizerError):
    pass


def _map_native(e: N.NativeError) -> TokenizerError:
    if e.code in (N.EINVAL, N.EILSEQ, N.ENOSPC):
        return InvalidInput(str(e))
    if e.code == N.ENOENT:
        return VocabNotFound(str(e))
    if e.code in (N.ENODEV, N.ENOMEM):
        return ServiceUnavailable(str(e))
    return Internal(str(e))


# --------------------------------------------------------------------------- boundary types
@dataclass(frozen=True)
class SecurityContext:
    """libs/modkit-security/src/context.rs:23-39 (tenant identity carried on every plugin call)"""
    subject_id: uuid.UUID
    subject_tenant_id: uuid.UUID
    subject_type: Optional[str] = None
    token_scopes: Sequence[str] = ()

    @staticmethod
    def anonymous() -> "SecurityContext":
        z = uuid.UUID(int=0)
        return SecurityContext(z, z, "service", ("*",))


@dataclass(frozen=True)
class VocabRef:
    """names a loaded vocabulary: registry name ("cl100k_base") or canonical model id ("openai::gpt-4")"""
    name: str


@dataclass
class EncodeBatchRequest:
    vocab: VocabRef
    bytes: np.ndarray            # uint8, packed UTF-8 of all prompts
    offsets: np.ndarray          # uint64, n+1, offsets[0] == 0
    vocabs_per_prompt: Optional[Sequence[VocabRef]] = None   # multi-tenant batches: one vocab per prompt
    vocab_index: Optional[np.ndarray] = None   # uint8, n: with it, vocabs_per_prompt lists the DISTINCT vocabularies and
                                               # vocab_index[i] picks prompt i's (large batches: no per-prompt objects)


@dataclass
class EncodeBatchResponse:
    ids: np.ndarray              # uint32 dense id stream
    offsets: np.ndarray          # uint64, n+1
    counts: np.ndarray           # uint32, n


@dataclass
class CountTokensRequest:
    vocab: VocabRef
    bytes: np.ndarray
    offsets: np.ndarray
    vocabs_per_prompt: Optional[Sequence[VocabRef]] = None
    vocab_index: Optional[np.ndarray] = None


@dataclass
class TruncateBatchRequest:
    """every prompt cut to k_i = min(count_i, budgets[i], max_tokens) tokens: its first k_i (keep="head") or its last (keep="tail")"""
    vocab: VocabRef
    bytes: np.ndarray
    offsets: np.ndarray
    max_tokens: int                          # L >= 1: ids per row
    keep: str = "head"                       # "head" | "tail"
    pad_id: int = 0
    budgets: Optional[np.ndarray] = None     # uint32, n, or None (max_tokens for every prompt)
    want_ids: bool = True                    # False: kept counts and cuts only, no id leaves the device
    vocabs_per_prompt: Optional[Sequence[VocabRef]] = None
    vocab_index: Optional[np.ndarray] = None


@dataclass
class TruncateBatchResponse:
    rows: Optional[np.ndarray]   # uint32 [n, max_tokens]: row i = its kept ids left-aligned, then pad_id; None without want_ids
    kept: np.ndarray             # uint32, n: k_i
    counts: np.ndarray           # uint32, n: the untruncated counts
    cut: np.ndarray              # uint64, n: byte offset of the cut inside prompt i (head: the kept text is prompt[:cut], tail: prompt[cut:])


@dataclass
class DecodeBatchRequest:
    vocab: VocabRef
    ids: np.ndarray              # uint32, packed ids of all sequences
    offsets: np.ndarray          # uint64, n+1 (in ids)
    vocabs_per_prompt: Optional[Sequence[VocabRef]] = None
    vocab_index: Optional[np.ndarray] = None


@dataclass
class DecodeBatchResponse:
    bytes: np.ndarray            # uint8, the sequences' bytes back to back (tiktoken decode_bytes; not necessarily valid UTF-8)
    offsets: np.ndarray          # uint64, n+1


@dataclass
class Usage:
    """gts.x.llmgw.core.usage.v1~"""
    input_tokens: int
    output_tokens: int = 0


@dataclass(frozen=True)
class ChatTemplate:
    """How a provider frames a list of chat messages into the token stream it bills as `Usage.input_tokens`
    (SURVEY.md section 8(f) item 2: "chat-template overhead accounting").  Two kinds:

    "overhead"  a fixed number of framing tokens a message (OpenAI's ChatML accounting: every message is
                <|start|>{role/name}\n{content}<|end|>\n = `tokens_per_message` tokens beside role and content, a `name` costs
                `tokens_per_name` more, the reply is primed with `reply_priming` tokens);
    "rendered"  the conversation is rendered to text around control tokens (Llama 3, Mistral): `bos`, then per message
                `message_prefix.format(role=...)` + content + `message_suffix`, then `generation_prompt`; the strings in
                `special_tokens` count one token each, the text between them is tokenised as ordinary text.

    Message CONTENT is always ordinary text: a message that spells a control token gets the pieces of that spelling, never the
    control token (the gateway does not let user text forge framing)."""
    kind: str = "overhead"
    tokens_per_message: int = 3
    tokens_per_name: int = 1
    reply_priming: int = 3
    bos: str = ""
    message_prefix: str = ""
    message_suffix: str = ""
    generation_prompt: str = ""
    special_tokens: Tuple[str, ...] = ()


# templates of the model families the stand-in vocabularies cover; a deployment lists its own next to the model's tokenizer
# (docs/model-registry-tokenizer-proposal.md)
CHAT_TEMPLATES = {
    # https://cookbook.openai.com "How to count tokens with tiktoken": gpt-3.5-turbo-0613 / gpt-4 and later
    "openai-chatml": ChatTemplate("overhead", tokens_per_message=3, tokens_per_name=1, reply_priming=3),
    # Meta Llama 3 instruct
    "llama3-instruct": ChatTemplate("rendered", bos="<|begin_of_text|>",
                                    message_prefix="<|start_header_id|>{role}<|end_header_id|>\n\n", message_suffix="<|eot_id|>",
                                    generation_prompt="<|start_header_id|>assistant<|end_header_id|>\n\n",
                                    special_tokens=("<|begin_of_text|>", "<|start_header_id|>", "<|end_header_id|>", "<|eot_id|>")),
}


# --------------------------------------------------------------------------- plugin trait
class TokenizerPluginClient:
    """plugin API (scoped in ClientHub by GTS instance id)"""

    def encode_batch(self, ctx: SecurityContext, req: EncodeBatchRequest) -> EncodeBatchResponse:
        raise NotImplementedError

    def count_tokens(self, ctx: SecurityContext, req: CountTokensRequest) -> np.ndarray:
        raise NotImplementedError

    def decode_batch(self, ctx: SecurityContext, req: "DecodeBatchRequest") -> "DecodeBatchResponse":
        raise NotImplementedError

    def truncate_batch(self, ctx: SecurityContext, req: "TruncateBatchRequest") -> "TruncateBatchResponse":
        raise NotImplementedError


GTS_PLUGIN_SCHEMA = "gts.x.core.modkit.plugin.v1~x.llmgw.tokenizer.plugin.v1~"


@dataclass
class PluginInstance:
    """BaseModkitPluginV1 content (libs/modkit/src/gts/plugin.rs:12-17)"""
    id: str
    vendor: str
    priority: int
    properties: dict = field(default_factory=dict)


class ClientHub:
    """type+scope keyed registry (libs/modkit/src/client_hub.rs:142-234), reduced to what the path needs"""

    def __init__(self):
        self._lock = threading.RLock()
        self._scoped: Dict[tuple, object] = {}

    def register_scoped(self, iface: type, scope: str, client: object) -> None:
        with self._lock:
            self._scoped[(iface, scope)] = client

    def get_scoped(self, iface: type, scope: str):
        with self._lock:
            try:
                return self._scoped[(iface, scope)]
            except KeyError:
                raise KeyError("ScopedNotFound(%s, %s)" % (iface.__name__, scope)) from None

    def try_get_scoped(self, iface: type, scope: str):
        with self._lock:
            return self._scoped.get((iface, scope))


def choose_plugin_instance(vendor: str, instances: Sequence[PluginInstance]) -> str:
    """vendor match, lowest priority wins, first wins ties (libs/modkit/src/plugins/mod.rs:136-191)"""
    best = None
    for inst in instances:
        if inst.vendor != vendor:
            continue
        if best is None or inst.priority < best.priority:
            best = inst
    if best is None:
        raise NoPluginAvailable("no tokenizer plugin for vendor %r" % vendor)
    return best.id


# --------------------------------------------------------------------------- the GPU plugin
class GpuBpeTokenizerPlugin(TokenizerPluginClient):
    """`gpu-bpe-tokenizer-plugin`: owns one device context; init = Module::init of the plugin
    (cuda context, vocab load -> device tables; multi-GPU broadcast is in cfbpe.dist)."""

    VENDOR = "cyberfabric"

    def __init__(self, device: int = 0, vocab_names: Sequence[str] = ("cl100k_base",), max_batch_bytes: int = 0,
                 max_prompts: int = 0, priority: int = 10, import_blobs: Optional[Dict[str, np.ndarray]] = None,
                 allow_stand_in: bool = False, devices: Optional[Sequence[int]] = None, n_workspaces: int = 1):
        """allow_stand_in: see cfbpe.vocabs.resolve -- benchmarks and tests only; a production plugin fails with VocabNotFound
        when a real rank file is missing instead of counting tokens with another vocabulary"""
        self.allow_stand_in = allow_stand_in
        self.max_batch_bytes = int(max_batch_bytes) if max_batch_bytes else 256 << 20     # cfbpe_create's defaults
        self.max_prompts = int(max_prompts) if max_prompts else 1 << 20
        try:
            self.ctx = N.Context(device, max_batch_bytes, max_prompts, devices=devices, n_workspaces=n_workspaces)
        except N.NativeError as e:
            raise _map_native(e) from e
        self._slot: Dict[str, int] = {}
        self.resolved: Dict[str, V.ResolvedVocab] = {}
        self._lock = threading.Lock()
        self.instance = PluginInstance(
            id=GTS_PLUGIN_SCHEMA + "cyberfabric.gpu_bpe.b200.v1", vendor=self.VENDOR, priority=priority,
            properties={"devices": list(devices) if devices else [device], "workspaces": n_workspaces, "vocabs": {}})
        for name in vocab_names:
            self.load_vocab(name, None if import_blobs is None else import_blobs.get(name))

    # -- vocab management (model-registry vocab loader side)
    def load_vocab(self, name: str, blob: Optional[np.ndarray] = None) -> int:
        with self._lock:
            if name in self._slot:
                return self._slot[name]
            slot = len(self._slot)
            if slot >= N.MAX_VOCABS:
                raise InvalidInput("too many vocabularies loaded")
            try:
                rv = V.resolve(name, self.allow_stand_in)
            except V.VocabUnavailable as e:
                raise VocabNotFound(str(e)) from e
            try:
                if blob is not None:
                    self.ctx.vocab_import(slot, blob)
                else:
                    self.ctx.vocab_load(slot, rv.file_bytes, rv.spec.fmt, rv.pattern_id, rv.max_ranks)
            except N.NativeError as e:
                raise _map_native(e) from e
            self._slot[name] = slot
            self.resolved[name] = rv
            # what a registry / operator sees about this instance: which file each vocabulary really is
            self.instance.properties["vocabs"][name] = {"slot": slot, "label": rv.label, "stand_in": rv.stand_in, "sha256": rv.sha256}
            return slot

    def export_vocab(self, name: str) -> np.ndarray:
        return self.ctx.vocab_export(self._slot[name])

    def _resolve_slot(self, ref: VocabRef) -> int:
        name = ref.name
        if name not in self._slot and name in V.MODEL_VOCABS:
            name = V.MODEL_VOCABS[name]
        if name not in self._slot:
            raise VocabNotFound("vocab %r is not loaded on this plugin" % ref.name)
        return self._slot[name]

    def _vocab_ids(self, req) -> Optional[np.ndarray]:
        n = len(req.offsets) - 1
        if req.vocabs_per_prompt is None:
            slot = self._resolve_slot(req.vocab)
            return None if slot == 0 else np.full(max(n, 1), slot, dtype=np.uint8)
        idx = getattr(req, "vocab_index", None)
        if idx is not None:         # a table of distinct vocabularies + one index per prompt
            if not isinstance(idx, np.ndarray) or idx.dtype != np.uint8 or idx.ndim != 1 or len(idx) != n:
                raise InvalidInput("vocab_index must be a uint8 array with one entry per prompt")
            lut = np.fromiter((self._resolve_slot(r) for r in req.vocabs_per_prompt), dtype=np.uint8, count=len(req.vocabs_per_prompt))
            if n and int(idx.max()) >= len(lut):
                raise InvalidInput("vocab_index names entry %d of %d vocabularies" % (int(idx.max()), len(lut)))
            return lut[idx] if n else np.zeros(1, dtype=np.uint8)
        if len(req.vocabs_per_prompt) != n:
            raise InvalidInput("vocabs_per_prompt must name one vocab per prompt")
        memo = {}
        out = np.empty(max(n, 1), dtype=np.uint8)
        for i, r in enumerate(req.vocabs_per_prompt):
            k = r.name
            v = memo.get(k)
            if v is None:
                v = memo[k] = self._resolve_slot(r)
            out[i] = v
        return out

    @staticmethod
    def _check_arrays(req):
        """what the C ABI cannot check (it takes no buffer lengths): dtypes, contiguity, and that the last offset stays
        inside the byte buffer -- otherwise the upload would read past the caller's array"""
        b, o = req.bytes, req.offsets
        if not isinstance(b, np.ndarray) or not isinstance(o, np.ndarray) or b.dtype != np.uint8 or o.dtype != np.uint64 or o.ndim != 1 or len(o) < 1:
            raise InvalidInput("bytes must be uint8 and offsets uint64 with n+1 entries")
        if not b.flags.c_contiguous or not o.flags.c_contiguous or b.ndim != 1:
            raise InvalidInput("bytes and offsets must be C-contiguous 1-D arrays")
        if int(o[0]) != 0 or int(o[-1]) > b.size:
            raise InvalidInput("offsets[0] must be 0 and offsets[n] (%d) must not exceed len(bytes) (%d)" % (int(o[-1]), b.size))

    # -- TokenizerPluginClient
    def encode_batch(self, ctx: SecurityContext, req: EncodeBatchRequest, out: Optional[EncodeBatchResponse] = None) -> EncodeBatchResponse:
        self._check_arrays(req)
        vid = self._vocab_ids(req)
        try:
            ids, offs, counts = self.ctx.encode_batch(
                req.bytes, req.offsets, vid,
                None if out is None else out.ids, None if out is None else out.offsets,
                None if out is None else out.counts)
        except N.NativeError as e:
            raise _map_native(e) from e
        return EncodeBatchResponse(ids, offs, counts)

    def count_tokens(self, ctx: SecurityContext, req: CountTokensRequest, out_counts: Optional[np.ndarray] = None) -> np.ndarray:
        self._check_arrays(req)
        vid = self._vocab_ids(req)
        try:
            return self.ctx.count_batch(req.bytes, req.offsets, vid, out_counts)
        except N.NativeError as e:
            raise _map_native(e) from e

    def truncate_batch(self, ctx: SecurityContext, req: TruncateBatchRequest) -> TruncateBatchResponse:
        self._check_arrays(req)
        if req.keep not in N.KEEP:
            raise InvalidInput("keep must be 'head' or 'tail', not %r" % (req.keep,))
        vid = self._vocab_ids(req)
        try:
            rows, kept, counts, cut = self.ctx.encode_truncated(req.bytes, req.offsets, vid, max_tokens=req.max_tokens, keep=N.KEEP[req.keep],
                                                                pad_id=req.pad_id, budgets=req.budgets, want_ids=req.want_ids)
        except N.NativeError as e:
            raise _map_native(e) from e
        return TruncateBatchResponse(rows, kept, counts, cut)

    def decode_batch(self, ctx: SecurityContext, req: DecodeBatchRequest) -> DecodeBatchResponse:
        if req.ids.dtype != np.uint32 or req.offsets.dtype != np.uint64 or len(req.offsets) < 1:
            raise InvalidInput("ids must be uint32 and offsets uint64 with n+1 entries")
        if not req.ids.flags.c_contiguous or not req.offsets.flags.c_contiguous or int(req.offsets[-1]) > req.ids.size:
            raise InvalidInput("offsets[n] must not exceed len(ids); arrays must be C-contiguous")
        vid = self._vocab_ids(req)
        try:
            out, offs = self.ctx.decode_batch(req.ids, req.offsets, vid)
        except N.NativeError as e:
            raise _map_native(e) from e
        return DecodeBatchResponse(out, offs)

    def close(self):
        self.ctx.close()


# --------------------------------------------------------------------------- gateway side
def pack_texts(texts: Sequence[str]):
    """list[str] -> (uint8 packed bytes, uint64 offsets): the packed multi-tenant prompt buffer"""
    enc = [t.encode("utf-8") for t in texts]
    offs = np.zeros(len(enc) + 1, dtype=np.uint64)
    if enc:
        offs[1:] = np.cumsum([len(e) for e in enc], dtype=np.uint64)
    data = np.frombuffer(b"".join(enc), dtype=np.uint8) if enc else np.zeros(0, dtype=np.uint8)
    return data, offs


class LlmGatewayTokenizerService:
    """`llm-gateway::tokenizer` + `llm-gateway::usage::count_tokens`: the gateway-side domain service.
    Plugin resolution is lazy and cached (libs/modkit/src/plugins/mod.rs:44-78)."""

    def __init__(self, hub: ClientHub, instances: Sequence[PluginInstance], vendor: str = GpuBpeTokenizerPlugin.VENDOR):
        self._hub, self._instances, self._vendor = hub, list(instances), vendor
        self._resolved: Optional[str] = None
        self._lock = threading.Lock()

    def _plugin(self) -> TokenizerPluginClient:
        with self._lock:
            if self._resolved is None:
                self._resolved = choose_plugin_instance(self._vendor, self._instances)
        p = self._hub.try_get_scoped(TokenizerPluginClient, self._resolved)
        if p is None:
            raise ServiceUnavailable("tokenizer plugin %s is not registered yet" % self._resolved)
        return p

    def encode(self, ctx: SecurityContext, model: str, texts: Sequence[str]) -> List[np.ndarray]:
        data, offs = pack_texts(texts)
        r = self._plugin().encode_batch(ctx, EncodeBatchRequest(VocabRef(model), data, offs))
        return [r.ids[int(r.offsets[i]):int(r.offsets[i + 1])] for i in range(len(texts))]

    def count_tokens(self, ctx: SecurityContext, model: str, messages: Sequence[dict]) -> Usage:
        """Usage.input_tokens of one chat request = sum of len(encode_ordinary(text)) over its
        TextContent parts (SURVEY.md 8 a4); the provider's framing on top of that: count_chat_tokens."""
        texts = [part["text"] for m in messages for part in m.get("content", []) if part.get("type") == "text"]
        if not texts:
            return Usage(0)
        data, offs = pack_texts(texts)
        counts = self._plugin().count_tokens(ctx, CountTokensRequest(VocabRef(model), data, offs))
        return Usage(int(counts.sum()))

    def count_chat_tokens(self, ctx: SecurityContext, model: str, messages: Sequence[dict], template: ChatTemplate) -> Usage:
        """`Usage.input_tokens` of one chat request as the provider counts it: content AND framing (ChatTemplate).
        messages: [{"role": "user", "name": optional, "content": [{"type": "text", "text": ...}, ...]}, ...]; parts that are
        not text (images ...) are priced elsewhere.  Every stretch of text of the whole request goes to the device in ONE batch."""
        import re
        texts: List[str] = []
        fixed = 0
        if template.kind == "overhead":
            for m in messages:
                fixed += template.tokens_per_message
                texts.append(str(m.get("role", "")))
                if m.get("name"):
                    fixed += template.tokens_per_name
                    texts.append(str(m["name"]))
                texts.extend(part["text"] for part in m.get("content", []) if part.get("type") == "text")
            fixed += template.reply_priming
        elif template.kind == "rendered":
            cut = re.compile("|".join(re.escape(t) for t in sorted(template.special_tokens, key=len, reverse=True))) if template.special_tokens else None

            def framing(text, into):          # control tokens count one each; the text between them is returned in pieces
                n, last = 0, 0
                for mt in (cut.finditer(text) if cut else ()):
                    into.append(text[last:mt.start()]); last = mt.end(); n += 1
                into.append(text[last:])
                return n
            # a stretch of ordinary text runs from one control token to the next: framing text and content are tokenised TOGETHER
            # (the pre-tokenizer may join the framing's trailing line breaks with the content's leading spaces)
            run: List[str] = [""]
            def feed_framing(text):
                nonlocal fixed
                pieces: List[str] = []
                fixed += framing(text, pieces)
                run[-1] += pieces[0]
                for p in pieces[1:]:
                    run.append(p)
            feed_framing(template.bos)
            for m in messages:
                feed_framing(template.message_prefix.format(role=m.get("role", "")))
                run[-1] += "".join(part["text"] for part in m.get("content", []) if part.get("type") == "text")
                feed_framing(template.message_suffix)
            feed_framing(template.generation_prompt)
            texts = [t for t in run if t]
        else:
            raise InvalidInput("unknown chat template kind %r" % template.kind)
        texts = [t for t in texts if t]
        if not texts:
            return Usage(fixed)
        data, offs = pack_texts(texts)
        counts = self._plugin().count_tokens(ctx, CountTokensRequest(VocabRef(model), data, offs))
        return Usage(fixed + int(counts.sum()))

    def encode_with_special(self, ctx: SecurityContext, model: str, texts: Sequence[str], special_tokens: dict,
                            allowed_special=(), disallowed_special="all") -> List[np.ndarray]:
        """tiktoken's `Encoding.encode(text, allowed_special=..., disallowed_special=...)` (SURVEY.md section 8(f) item 2):
        the text is cut at every occurrence of an allowed special token (leftmost first), the stretches between them go
        through encode_ordinary -- all stretches of all texts in ONE plugin batch -- and the special ids are put back in.
        special_tokens: {"<|endoftext|>": 100257, ...}; allowed / disallowed: "all" or a set of token strings; a text
        that holds a disallowed special token raises InvalidInput (tiktoken raises ValueError).  Defaults as tiktoken's:
        nothing allowed, everything disallowed -- user text that spells a control token is refused, not turned into one."""
        import re
        allowed = set(special_tokens) if allowed_special == "all" else set(allowed_special)
        disallowed = (set(special_tokens) - allowed) if disallowed_special == "all" else set(disallowed_special)
        unknown = allowed - set(special_tokens)
        if unknown:
            raise InvalidInput("allowed special tokens without an id: %s" % sorted(unknown))
        if disallowed:
            bad = re.compile("|".join(re.escape(t) for t in sorted(disallowed, key=len, reverse=True)))
            for t in texts:
                m = bad.search(t)
                if m:
                    raise InvalidInput("the text holds the special token %r, which is not allowed here" % m.group())
        cut = re.compile("|".join(re.escape(t) for t in sorted(allowed, key=len, reverse=True))) if allowed else None
        plan, stretches = [], []          # per text: list of ("s", stretch index) | ("t", special id)
        for t in texts:
            steps, pos = [], 0
            for m in (cut.finditer(t) if cut else ()):
                if m.start() > pos:
                    steps.append(("s", len(stretches))); stretches.append(t[pos:m.start()])
                steps.append(("t", int(special_tokens[m.group()])))
                pos = m.end()
            if pos < len(t):
                steps.append(("s", len(stretches))); stretches.append(t[pos:])
            plan.append(steps)
        enc = self.encode(ctx, model, stretches) if stretches else []
        out = []
        for steps in plan:
            parts = [enc[i] if kind == "s" else np.array([i], dtype=np.uint32) for kind, i in steps]
            out.append(np.concatenate(parts).astype(np.uint32) if parts else np.zeros(0, dtype=np.uint32))
        return out

    def truncate(self, ctx: SecurityContext, model: str, texts: Sequence[str], max_tokens: int, keep: str = "head") -> List[Tuple[np.ndarray, int]]:
        """Each text cut to at most max_tokens tokens: its first ones (keep="head") or its last ones (keep="tail").  Returns per text
        (kept ids, byte cut): head keeps text.encode()[:cut], tail keeps text.encode()[cut:].
        Two caveats.  The kept ids are a slice of the text's full encoding, and re-encoding the kept bytes need not give the same
        ids: the pre-tokenizer's lookahead (\\s+(?!\\S)) sees different text at the cut.  And the cut is the token boundary as it is:
        byte-level tokens split CJK characters and emoji, so it can fall inside a multi-byte UTF-8 character (the kept bytes then
        do not decode as UTF-8 on their own)."""
        data, offs = pack_texts(texts)
        r = self._plugin().truncate_batch(ctx, TruncateBatchRequest(VocabRef(model), data, offs, max_tokens, keep))
        return [(r.rows[i, :int(r.kept[i])].copy(), int(r.cut[i])) for i in range(len(texts))]

    def check_budget(self, ctx: SecurityContext, model: str, messages: Sequence[dict], remaining_tokens: int) -> bool:
        """pre-call estimate used by check_budget (modules/llm-gateway/docs/DESIGN.md:833-855)"""
        return self.count_tokens(ctx, model, messages).input_tokens <= remaining_tokens


# --------------------------------------------------------------------------- micro-batcher (SURVEY.md section 8(f) item 4)
class CountTokensMicroBatcher:
    """Coalesces concurrent count_tokens calls (one chat request each, a few KB) into GPU-sized batches.

    The gateway's request handlers call `count(ctx, model, texts)` from many threads (tokio tasks behind spawn_blocking in the
    Rust host); a single worker drains the queue, packs what is waiting -- up to max_batch_bytes, or whatever arrived within
    max_wait_s of the first item -- into ONE CountTokensRequest with one vocabulary per prompt, and hands every caller its own
    counts.  In ModKit terms this is a `stateful` lifecycle task (docs/modkit_unified_system/08_lifecycle_stateful_tasks.md:14-58):
    start() / stop() are its hooks.  A failed batch fails exactly the calls that were in it."""

    def __init__(self, plugin: TokenizerPluginClient, max_batch_bytes: int = 8 << 20, max_wait_s: float = 0.0005, max_queue: int = 65536,
                 max_batch_prompts: int = 1 << 16):
        import queue
        # a batch never exceeds what the plugin's device context accepts (otherwise one oversize batch fails every caller in it)
        lim_b = getattr(plugin, "max_batch_bytes", None)
        lim_p = getattr(plugin, "max_prompts", None)
        self._max_bytes = int(min(max_batch_bytes, lim_b)) if lim_b else int(max_batch_bytes)
        self._max_prompts = int(min(max_batch_prompts, lim_p)) if lim_p else int(max_batch_prompts)
        self._plugin, self._max_wait = plugin, float(max_wait_s)
        self._q = queue.Queue(maxsize=max_queue)
        self._worker: Optional[threading.Thread] = None
        self._stop = threading.Event()
        self._carry = None        # an item that did not fit the batch being packed: first of the next one
        self.batches = 0          # how many plugin calls were made (for tests / metrics)
        self.items = 0

    def start(self):
        if self._worker is None:
            self._stop.clear()
            self._worker = threading.Thread(target=self._run, name="count-tokens-batcher", daemon=True)
            self._worker.start()
        return self

    def stop(self):
        self._stop.set()
        if self._worker is not None:
            self._q.put(None)
            self._worker.join()
            self._worker = None

    def count(self, ctx: SecurityContext, model: str, texts: Sequence[str], timeout: Optional[float] = None) -> np.ndarray:
        """token counts of `texts` under `model`'s vocabulary; blocks until the batch this call rode in is done.
        What can be checked per request is checked HERE, before the request joins a batch with other tenants' requests:
        an unknown model or an oversize request fails this caller only."""
        import queue
        if self._worker is None:
            raise ServiceUnavailable("the micro-batcher is not running")
        enc = [t.encode("utf-8") for t in texts]
        size = sum(len(t) for t in enc)
        if size > self._max_bytes or len(enc) > self._max_prompts:
            raise InvalidInput("the request (%d bytes, %d texts) exceeds the batch limits (%d bytes, %d prompts)"
                               % (size, len(enc), self._max_bytes, self._max_prompts))
        resolve = getattr(self._plugin, "_resolve_slot", None)
        if resolve is not None:
            resolve(VocabRef(model))          # VocabNotFound for this caller alone
        item = {"ctx": ctx, "model": model, "texts": enc, "size": size, "done": threading.Event(), "out": None, "err": None}
        try:
            self._q.put(item, timeout=timeout)
        except queue.Full:
            raise ServiceUnavailable("the count_tokens queue is full") from None
        if not item["done"].wait(timeout):
            raise ServiceUnavailable("count_tokens timed out")
        if item["err"] is not None:
            raise item["err"]
        return item["out"]

    def _run(self):
        import queue, time
        while not self._stop.is_set():
            first = self._carry if self._carry is not None else self._q.get()
            self._carry = None
            if first is None:
                break
            batch, size, n = [first], first["size"], len(first["texts"])
            deadline = time.monotonic() + self._max_wait
            while size < self._max_bytes and n < self._max_prompts:
                try:
                    nxt = self._q.get(timeout=max(0.0, deadline - time.monotonic()))
                except queue.Empty:
                    break
                if nxt is None:
                    self._stop.set()
                    break
                if size + nxt["size"] > self._max_bytes or n + len(nxt["texts"]) > self._max_prompts:
                    self._carry = nxt          # does not fit: it opens the next batch
                    break
                batch.append(nxt)
                size += nxt["size"]
                n += len(nxt["texts"])
            self._flush(batch)
        if self._carry is not None:
            self._carry["err"] = ServiceUnavailable("the micro-batcher stopped"); self._carry["done"].set(); self._carry = None
        while True:               # fail what is still queued
            try:
                it = self._q.get_nowait()
            except queue.Empty:
                break
            if it is not None:
                it["err"] = ServiceUnavailable("the micro-batcher stopped"); it["done"].set()

    def _call(self, batch):
        """one plugin call for `batch`; fills out / raises"""
        pieces = [t for it in batch for t in it["texts"]]
        if not pieces:
            for it in batch:
                it["out"] = np.zeros(0, dtype=np.uint32)
            return
        offs = np.zeros(len(pieces) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(t) for t in pieces])
        data = np.frombuffer(b"".join(pieces), dtype=np.uint8)
        vocabs = [VocabRef(it["model"]) for it in batch for _ in it["texts"]]
        # the call carries the first request's SecurityContext only as the transport identity: counting tokens reads no
        # tenant-scoped state, and every caller gets exactly its own prompts' counts back
        counts = self._plugin.count_tokens(batch[0]["ctx"], CountTokensRequest(vocabs[0], data, offs, vocabs_per_prompt=vocabs))
        k = 0
        for it in batch:
            n = len(it["texts"])
            it["out"] = np.array(counts[k:k + n], dtype=np.uint32)
            k += n

    def _flush(self, batch):
        """A failed batch is retried request by request, so a bad request (malformed UTF-8, a model whose vocabulary was
        unloaded meanwhile) fails its own caller and nobody else's -- requests of different tenants share batches."""
        try:
            self._call(batch)
            self.batches += 1
        except TokenizerError:
            for it in batch:
                try:
                    self._call([it])
                except Exception as e:    # noqa: BLE001
                    it["err"] = e
                self.batches += 1
        except Exception as e:    # noqa: BLE001 -- not an input problem: every caller of this batch gets the error
            for it in batch:
                it["err"] = e
            self.batches += 1
        self.items += len(batch)
        for it in batch:
            it["done"].set()
