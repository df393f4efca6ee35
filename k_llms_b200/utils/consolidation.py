"""Consolidation glue: n choices -> align -> consensus -> choices[0] = consensus, choices[1..n] = originals.

Same four entry points, signatures and result shape as reference k_llms/utils/consolidation.py:63-493; the four
near-identical bodies there share one implementation here.  The consensus itself runs on the GPU
(`consensus_utils.consensus_values`); JSON parsing and object rebuilding stay host Python (SURVEY.md §8a a8).
"""
from __future__ import annotations

import asyncio
import json
from typing import Any, List, Optional, Union

from openai.types.chat import ChatCompletion, ChatCompletionMessage, ParsedChatCompletion
from openai.types.chat.chat_completion import Choice
from openai.types.chat.parsed_chat_completion import ParsedChatCompletionMessage, ParsedChoice
from pydantic import BaseModel

from ..types.completions import KLLMsChatCompletion
from ..types.parsed import KLLMsParsedChatCompletion
from .consensus_utils import (
    ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    ConsensusSettings,
    async_consensus_values,
    async_recursive_list_alignments,
    check_candidate_logprobs,
    consensus_values,
    recursive_list_alignments,
)


def _safe_parse_content(content: str) -> dict:
    """JSON if it parses, else {"text": content} (reference consolidation.py:25-38)."""
    try:
        return json.loads(content)
    except (json.JSONDecodeError, TypeError):
        return {"text": content}


def _format_consensus_content(consensus_content: Any) -> str:
    """Inverse of _safe_parse_content for the consensus message (reference consolidation.py:41-60)."""
    if consensus_content is None:
        return ""
    if isinstance(consensus_content, dict) and len(consensus_content) == 1 and isinstance(consensus_content.get("text"), str):
        return consensus_content["text"]
    return json.dumps(consensus_content)


def _contents_of(choices) -> List[dict]:
    return [_safe_parse_content(c.message.content) for c in choices if c.message.content]


def _logprobs_of(choices, settings) -> Optional[List[List[float]]]:
    """Under likelihood weighting, the token logprobs (choice.logprobs.content[*].logprob) of the choices _contents_of keeps: a
    dropped choice's logprobs are dropped with it.  None under uniform weighting."""
    if settings.candidate_weighting != "likelihood":
        return None
    kept = [c for c in choices if c.message.content]
    seqs = [[t.logprob for t in c.logprobs.content] if c.logprobs is not None and c.logprobs.content is not None else None
            for c in kept]
    return check_candidate_logprobs(settings, seqs, len(kept))


def _native_alignment(contents, settings):
    """The alignment pre-pass in native code (H2, `kc_align_json`: same result as `recursive_list_alignments`, pinned on the
    reference's goldens) — or None when the record needs the Python pre-pass: another similarity method than the default,
    string pairs that go to the embeddings service (both longer than 50 characters), non-ASCII text."""
    if settings.string_similarity_method != "embeddings":
        return None
    from .. import _native
    return _native.align_json(contents, settings.min_support_ratio)


def _native_settings(settings) -> bool:
    """The settings the native JSON path (H1, kc_consolidate_json) implements: the reference's defaults."""
    return (not settings.allow_none_as_candidate and settings.string_similarity_method == "embeddings"
            and settings.string_consensus_method == "centroid" and settings.min_support_ratio == 0.51)


def _consensus_of_choices_native(choices, settings, embed, logprobs=None):
    """The whole per-request path in native code (H1): the n `choice.message.content` texts in -> (consensus value,
    likelihoods), i.e. parse + alignment pre-pass + vote / numeric / medoid kernels + decode — or None when the request needs
    the Python path (non-default settings, fewer than two non-empty contents, anything H1 declines; no embeddings callable:
    the reference raises ValueError for primitive fields then, cu:1445-1446, and so does the Python path)."""
    from .. import _native
    if embed is None:
        return None
    texts = [c.message.content for c in choices if c.message.content]  # the filter of _contents_of (reference consolidation.py:92)
    if len(texts) < 2 or len(texts) > _native.MAX_CANDIDATES or not _native_settings(settings):
        return None
    out = _combiner.run(texts, settings.rel_eps, settings.abs_eps, logprobs)
    if out is None:
        return None
    content_text, likelihoods_text = out
    try:  # undo _format_consensus_content: a consensus that is not a JSON object is the unwrapped {"text": s}
        value = json.loads(content_text)
    except ValueError:
        value = None
    if not isinstance(value, dict):
        value = {"text": content_text}
    return value, json.loads(likelihoods_text)


def _native_consolidate(records, rel_eps, abs_eps, device: int = 0, logprobs=None):
    """records of n candidate texts -> [(content, likelihoods text) or None]: the device JSON path (H1g,
    kc_consolidate_json_packed: scan / key sort / typing / encode / K1 + K2 / emit on the GPU; re-entrant, pooled streams), which
    hands what it does not model to the host path (H1, kc_consolidate_json) inside the same call.  logprobs[r][c] = the token
    logprobs of records[r][c]: the likelihood-weighted entry (kc_consolidate_json_packed_weighted), which has no host path — what
    the device declines comes back as None."""
    import numpy as np

    from .. import _native
    pinned = len(records) >= 256  # page-locking only pays for batches
    blob, off, n = _native.pack_texts(records, pinned=pinned)
    lp = None
    if logprobs is not None:
        lp = _native.pack_logprobs(logprobs, pinned=pinned)
        if np.isnan(lp[0][:lp[1][-1]]).any():
            raise ValueError("candidate_weighting='likelihood': a candidate has a NaN logprob")
    res = _native.consolidate_json_packed(blob, off, n, rel_eps, abs_eps, device, logprobs=lp)
    try:
        return res.pairs()
    finally:
        res.close()


class _Combiner:
    """Per-request consolidations that arrive while another one is on the GPU are COMBINED into one batched call (flat
    combining: the thread that holds the device runs its own request, then everything that queued up meanwhile as one
    kc_consolidate_json_packed call, and hands the results back).  An idle caller pays nothing (it takes the device and runs
    directly); under load the cost per request falls from one launch sequence each (~0.5 ms) towards the batched rate
    (tools/latency.py: tens of thousands of requests per second)."""

    def __init__(self):
        import threading
        self._device = threading.Lock()
        self._qlock = threading.Lock()
        self._queue: list = []

    def _drain(self):
        while True:
            with self._qlock:
                batch, self._queue = self._queue, []
            if not batch:
                return
            groups: dict = {}
            for item in batch:  # one call per candidate count, eps and weighting
                groups.setdefault((len(item["texts"]), item["eps"], item["lp"] is not None), []).append(item)
            for (_n, eps, weighted), items in groups.items():
                try:
                    outs = _native_consolidate([it["texts"] for it in items], eps[0], eps[1],
                                               logprobs=[it["lp"] for it in items] if weighted else None)
                    for it, o in zip(items, outs):
                        it["out"] = o
                except BaseException as exc:  # hand the failure to every waiter of the group
                    for it in items:
                        it["err"] = exc
                for it in items:
                    it["done"].set()

    def run(self, texts, rel_eps, abs_eps, logprobs=None):
        import threading
        item = {"texts": texts, "eps": (rel_eps, abs_eps), "lp": logprobs, "done": threading.Event(), "out": None, "err": None}
        with self._qlock:
            self._queue.append(item)
        while not item["done"].is_set():
            if self._device.acquire(blocking=False):
                try:
                    self._drain()
                finally:
                    self._device.release()
            else:
                item["done"].wait(0.0005)
        if item["err"] is not None:
            raise item["err"]
        return item["out"]


_combiner = _Combiner()


def _check_candidates(n: int) -> None:
    from .. import _native
    if n > _native.MAX_CANDIDATES:
        raise ValueError(f"{n} candidates in one request: k_llms_b200 consolidates at most {_native.MAX_CANDIDATES} "
                         "(README.md, Limits)")


def _consensus_sync(contents, settings, embed, client, logprobs=None):
    if len(contents) >= 2:  # reference consolidation.py:96-104
        aligned = _native_alignment(contents, settings)
        if aligned is None:
            aligned, _ = recursive_list_alignments(contents, settings.string_similarity_method, embed, client, settings.min_support_ratio)
        contents = [(d if isinstance(d, dict) else {}) for d in aligned]
    return consensus_values(contents, settings, embed, client=client, candidate_logprobs=logprobs)


async def _consensus_async(contents, settings, embed, client, logprobs=None):
    if len(contents) >= 2:
        aligned = _native_alignment(contents, settings)
        if aligned is None:
            aligned, _ = await async_recursive_list_alignments(contents, settings.string_similarity_method, embed, client,
                                                               settings.min_support_ratio)
        contents = [(d if isinstance(d, dict) else {}) for d in aligned]
    return await async_consensus_values(contents, settings, embed, client=client, candidate_logprobs=logprobs)


def _assemble_plain(base: ChatCompletion, heads, consensus_content, likelihoods) -> KLLMsChatCompletion:
    """heads: the choices whose message/finish_reason/logprobs become choices[1..]; heads[0] lends its
    function_call / tool_calls / refusal / finish_reason / logprobs to the consensus choice."""
    first = heads[0] if heads else None
    message = ChatCompletionMessage(
        role="assistant",
        content=_format_consensus_content(consensus_content),
        function_call=first.message.function_call if first else None,
        tool_calls=first.message.tool_calls if first else None,
        refusal=first.message.refusal if first else None,
    )
    consensus_choice = Choice(finish_reason=first.finish_reason if first else "stop", index=0, message=message,
                              logprobs=first.logprobs if first else None)
    originals = [Choice(finish_reason=c.finish_reason, index=i + 1, message=c.message, logprobs=c.logprobs)
                 for i, c in enumerate(heads)]
    return KLLMsChatCompletion.model_validate(
        {**base.model_dump(), "choices": [consensus_choice] + originals, "likelihoods": likelihoods, "usage": base.usage})


def consolidate_chat_completions(
    completions: Union[List[ChatCompletion], ChatCompletion],
    get_openai_embeddings_from_text: SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    consensus_settings: ConsensusSettings = ConsensusSettings(),
) -> KLLMsChatCompletion:
    """One ChatCompletion with n choices, or a list of completions (reference consolidation.py:63-216)."""
    if isinstance(completions, ChatCompletion):
        completion = completions
        assert len(completion.choices) > 0, "Cannot consolidate empty list of choices"
        if len(completion.choices) == 1:
            return KLLMsChatCompletion.model_validate(completion.model_dump())
        _check_candidates(len(completion.choices))
        lps = _logprobs_of(completion.choices, consensus_settings)
        content, likelihoods = (_consensus_of_choices_native(completion.choices, consensus_settings, get_openai_embeddings_from_text, lps)
                                or _consensus_sync(_contents_of(completion.choices), consensus_settings, get_openai_embeddings_from_text, client,
                                                   lps))
        return _assemble_plain(completion, list(completion.choices), content, likelihoods)
    completion_list = completions
    assert len(completion_list) > 0, "Cannot consolidate empty list of completions"
    if len(completion_list) == 1:
        return KLLMsChatCompletion.model_validate(completion_list[0].model_dump())
    _check_candidates(len(completion_list))
    # choices[i + 1] keeps the index of completion i and completion_list[0] lends its head fields (reference consolidation.py:
    # 176-216); a completion without choices contributes nothing
    firsts = [(i, c.choices[0]) for i, c in enumerate(completion_list) if c.choices]
    heads = [c for _, c in firsts]
    lps = _logprobs_of(heads, consensus_settings)
    content, likelihoods = (_consensus_of_choices_native(heads, consensus_settings, get_openai_embeddings_from_text, lps)
                            or _consensus_sync(_contents_of(heads), consensus_settings, get_openai_embeddings_from_text, client, lps))
    out = _assemble_plain(completion_list[0], heads, content, likelihoods)
    for k, (i, _) in enumerate(firsts):
        out.choices[k + 1].index = i + 1
    return out


async def async_consolidate_chat_completions(
    completion: ChatCompletion,
    async_get_openai_embeddings_from_text: ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    consensus_settings: ConsensusSettings = ConsensusSettings(),
) -> KLLMsChatCompletion:
    """Reference consolidation.py:219-303."""
    assert len(completion.choices) > 0, "Cannot consolidate empty list of choices"
    if len(completion.choices) == 1:
        return KLLMsChatCompletion.model_validate(completion.model_dump())
    _check_candidates(len(completion.choices))
    # the native JSON paths implement the SYNC semantics; the reference's async dispatcher differs on numeric fields
    # (cu:1638-1688: no clustering), so the async entry points plan in Python (async_consensus_values) — votes still on the GPU
    content, likelihoods = await _consensus_async(_contents_of(completion.choices), consensus_settings,
                                                  async_get_openai_embeddings_from_text, client,
                                                  _logprobs_of(completion.choices, consensus_settings))
    return _assemble_plain(completion, list(completion.choices), content, likelihoods)


def _assemble_parsed(completion: ParsedChatCompletion, consensus_content, likelihoods, response_format, keep_usage: bool):
    parsed = None
    if response_format and consensus_content is not None:
        try:  # validation failures are swallowed: parsed stays None (reference consolidation.py:358-365)
            if isinstance(response_format, type) and issubclass(response_format, BaseModel):
                parsed = response_format.model_validate(consensus_content)
        except Exception:
            parsed = None
    first = completion.choices[0]
    message = ParsedChatCompletionMessage(
        role="assistant",
        content=_format_consensus_content(consensus_content),
        function_call=first.message.function_call,
        tool_calls=first.message.tool_calls,
        refusal=first.message.refusal,
        parsed=parsed,
    )
    consensus_choice = ParsedChoice(finish_reason=first.finish_reason, index=0, message=message, logprobs=first.logprobs)
    originals = [ParsedChoice(finish_reason=c.finish_reason, index=i + 1, message=c.message, logprobs=c.logprobs)
                 for i, c in enumerate(completion.choices)]
    payload = {**completion.model_dump(), "choices": [consensus_choice] + originals, "likelihoods": likelihoods}
    if keep_usage:
        payload["usage"] = completion.usage
    return KLLMsParsedChatCompletion.model_validate(payload)


def consolidate_parsed_chat_completions(
    completion: ParsedChatCompletion,
    get_openai_embeddings_from_text: SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    consensus_settings: ConsensusSettings = ConsensusSettings(),
    response_format: Optional[type] = None,
) -> KLLMsParsedChatCompletion:
    """Reference consolidation.py:306-399."""
    assert len(completion.choices) > 0, "Cannot consolidate empty list of choices"
    if len(completion.choices) == 1:
        return KLLMsParsedChatCompletion.model_validate(completion.model_dump())
    _check_candidates(len(completion.choices))
    lps = _logprobs_of(completion.choices, consensus_settings)
    content, likelihoods = (_consensus_of_choices_native(completion.choices, consensus_settings, get_openai_embeddings_from_text, lps)
                            or _consensus_sync(_contents_of(completion.choices), consensus_settings, get_openai_embeddings_from_text, client,
                                               lps))
    return _assemble_parsed(completion, content, likelihoods, response_format, keep_usage=True)


async def async_consolidate_parsed_chat_completions(
    completion: ParsedChatCompletion,
    async_get_openai_embeddings_from_text: ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    consensus_settings: ConsensusSettings = ConsensusSettings(),
    response_format: Optional[type] = None,
) -> KLLMsParsedChatCompletion:
    """Reference consolidation.py:402-493 (the reference's async twin does not re-attach `usage`; model_dump keeps it)."""
    assert len(completion.choices) > 0, "Cannot consolidate empty list of choices"
    if len(completion.choices) == 1:
        return KLLMsParsedChatCompletion.model_validate(completion.model_dump())
    _check_candidates(len(completion.choices))
    content, likelihoods = await _consensus_async(_contents_of(completion.choices), consensus_settings,
                                                  async_get_openai_embeddings_from_text, client,
                                                  _logprobs_of(completion.choices, consensus_settings))
    return _assemble_parsed(completion, content, likelihoods, response_format, keep_usage=False)


def consolidate_contents_batch(records: List[List[str]], consensus_settings: ConsensusSettings = ConsensusSettings(),
                               get_openai_embeddings_from_text: Optional[SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE] = None,
                               client: Any = None, device: int = 0, logprobs: Optional[List[List[List[float]]]] = None):
    """Batched consolidation of raw contents (new; the reference has no batch dimension): for every record, the n
    `choice.message.content` strings in -> (consensus content string, likelihoods) out, exactly what the per-request
    functions above put into choices[0] and `likelihoods`.

    With the default settings the batch goes to the device JSON path (H1g, kc_consolidate_json_packed: the texts are copied to
    the GPU as they are; scan / key sort / typing / encode / K1 + K2 / emit run there); records that path does not model
    (nested objects, lists, multi-word strings, escapes, ...) are consolidated by the native host path (H1: C++ parse /
    alignment pre-pass / encode / decode + K1/K2/K4) inside the same call, and what that declines too (a key mixing objects
    with other types, string pairs that need the embeddings service, non-ASCII text, ...) takes the Python + GPU path.

    With consensus_settings.candidate_weighting == "likelihood", logprobs[r][c] = the token logprobs of records[r][c] (one sequence
    per text, empty texts included: their logprobs are dropped with them).  The batch goes to the weighted device entry
    (kc_consolidate_json_packed_weighted); what it declines takes the weighted Python + GPU path (there is no weighted host path)."""
    from .. import _native
    default_eps = (consensus_settings.rel_eps, consensus_settings.abs_eps)
    native: List[Any] = [None] * len(records)
    weighted = consensus_settings.candidate_weighting == "likelihood"
    if weighted:
        if logprobs is None:
            raise ValueError("candidate_weighting='likelihood' needs logprobs: one list of token logprobs per candidate text")
        if len(logprobs) != len(records) or any(lp is None or len(lp) != len(texts) for lp, texts in zip(logprobs, records)):
            raise ValueError("candidate_weighting='likelihood': logprobs must hold one sequence per candidate text of every record")
    if _native_settings(consensus_settings):
        by_n: dict = {}
        for i, texts in enumerate(records):
            if len(texts) >= 2:
                by_n.setdefault(len(texts), []).append(i)
        for n, idxs in by_n.items():
            _check_candidates(n)
            outs = _native_consolidate([records[i] for i in idxs], default_eps[0], default_eps[1], device,
                                       [logprobs[i] for i in idxs] if weighted else None)
            for i, o in zip(idxs, outs):
                native[i] = o
    results = []
    embed = get_openai_embeddings_from_text if get_openai_embeddings_from_text is not None else (lambda texts: [[0.0] for _ in texts])
    for i, (texts, nat) in enumerate(zip(records, native)):
        if nat is not None:
            results.append((nat[0], json.loads(nat[1])))
            continue
        contents = [_safe_parse_content(t) for t in texts if t]
        lps = check_candidate_logprobs(consensus_settings, [lp for t, lp in zip(texts, logprobs[i]) if t], len(contents)) if weighted else None
        _check_candidates(len(contents))
        if len(texts) == 1:  # a single choice is returned as it is (reference consolidation.py:85-87)
            results.append((texts[0], None))
            continue
        # one non-empty content among several choices still goes through consensus_values, like the per-request path
        value, likelihoods = _consensus_sync(contents, consensus_settings, embed, client, lps)
        results.append((_format_consensus_content(value), likelihoods))
    return results
