"""`.chat.completions.create()` / `.parse()` for the sync and async wrappers
(reference k_llms/resources/completions/completions.py:15-294): forward the request to OpenAI with `n`, then
consolidate the n choices.  Keyword surface and defaults are the reference's, plus `consensus_settings` (this package's own:
e.g. ConsensusSettings(candidate_weighting="likelihood"), which asks the API for the choices' token logprobs)."""
from __future__ import annotations

from typing import TYPE_CHECKING, Any, List, Optional, Union

from ...types.completions import KLLMsChatCompletion
from ...types.parsed import KLLMsParsedChatCompletion
from ...utils.consensus_utils import ConsensusSettings
from ...utils.consolidation import (
    async_consolidate_chat_completions,
    async_consolidate_parsed_chat_completions,
    consolidate_chat_completions,
    consolidate_parsed_chat_completions,
)

if TYPE_CHECKING:  # pragma: no cover
    from ...client import AsyncKLLMs, KLLMs

_SAMPLING_KEYS = ("temperature", "max_tokens", "top_p", "frequency_penalty", "presence_penalty", "stop", "seed")
_EMBED_MODEL, _EMBED_BATCH = "text-embedding-3-small", 2048


MAX_N = 64  # _native.MAX_CANDIDATES: one kernel row per field holds every candidate; there is no CPU path to fall back to


def _call_params(base: dict, sampling: dict, n: Optional[int], extra: dict, settings: Optional[ConsensusSettings] = None) -> dict:
    if n is not None and n > MAX_N:  # fail BEFORE the (paid) API call: the n choices could not be consolidated
        raise ValueError(f"n={n}: k_llms_b200 consolidates at most {MAX_N} candidates per request (README.md, Limits)")
    likelihood = settings is not None and settings.candidate_weighting == "likelihood"
    if likelihood and extra.get("logprobs", True) is False:  # likewise: the choices could not be weighted
        raise ValueError("candidate_weighting='likelihood' weights the choices by their token logprobs: it cannot be combined "
                         "with logprobs=False")
    params = dict(base)
    params.update({k: v for k, v in sampling.items() if v is not None})
    params.update(extra)
    if likelihood:
        params["logprobs"] = True
    if n and n > 1:  # OpenAI's native n: all candidates come back in one response
        params["n"] = n
    return params


class Completions:
    def __init__(self, wrapper: "KLLMs"):
        self._wrapper = wrapper

    def _embed(self, texts: List[str]) -> List[List[float]]:
        return self._wrapper.get_embeddings(texts, _EMBED_MODEL, _EMBED_BATCH, False)

    def create(self, *, messages: List[Any], model: str, n: Optional[int] = None, temperature: Optional[float] = None,
               max_tokens: Optional[int] = None, top_p: Optional[float] = None, frequency_penalty: Optional[float] = None,
               presence_penalty: Optional[float] = None, stop: Optional[Union[str, List[str]]] = None,
               seed: Optional[int] = None, response_format: Any = None, consensus_settings: Optional[ConsensusSettings] = None,
               **kwargs: Any) -> KLLMsChatCompletion:
        kwargs.pop("stream", None)  # streaming is not supported: always stream=False
        settings = consensus_settings or ConsensusSettings()
        sampling = dict(temperature=temperature, max_tokens=max_tokens, top_p=top_p, frequency_penalty=frequency_penalty,
                        presence_penalty=presence_penalty, stop=stop, seed=seed, response_format=response_format)
        params = _call_params({"messages": messages, "model": model, "stream": False}, sampling, n, kwargs, settings)
        completion = self._wrapper.client.chat.completions.create(**params)
        return consolidate_chat_completions(completion, self._embed, client=self._wrapper.client, consensus_settings=settings)

    def parse(self, *, messages: List[Any], model: str, response_format: Any, n: Optional[int] = None,
              temperature: Optional[float] = None, max_tokens: Optional[int] = None, top_p: Optional[float] = None,
              frequency_penalty: Optional[float] = None, presence_penalty: Optional[float] = None,
              stop: Optional[Union[str, List[str]]] = None, seed: Optional[int] = None,
              consensus_settings: Optional[ConsensusSettings] = None, **kwargs: Any) -> KLLMsParsedChatCompletion:
        settings = consensus_settings or ConsensusSettings()
        sampling = dict(temperature=temperature, max_tokens=max_tokens, top_p=top_p, frequency_penalty=frequency_penalty,
                        presence_penalty=presence_penalty, stop=stop, seed=seed)
        params = _call_params({"messages": messages, "model": model, "response_format": response_format}, sampling, n, kwargs, settings)
        completion = self._wrapper.client.beta.chat.completions.parse(**params)
        return consolidate_parsed_chat_completions(completion, self._embed, response_format=response_format,
                                                   client=self._wrapper.client, consensus_settings=settings)


class AsyncCompletions:
    def __init__(self, wrapper: "AsyncKLLMs"):
        self._wrapper = wrapper

    async def _embed(self, texts: List[str]) -> List[List[float]]:
        return await self._wrapper.get_embeddings(texts, _EMBED_MODEL, _EMBED_BATCH, False)

    async def create(self, *, messages: List[Any], model: str, response_format: Any = None, n: Optional[int] = None,
                     temperature: Optional[float] = None, max_tokens: Optional[int] = None, top_p: Optional[float] = None,
                     frequency_penalty: Optional[float] = None, presence_penalty: Optional[float] = None,
                     stop: Optional[Union[str, List[str]]] = None, seed: Optional[int] = None,
                     consensus_settings: Optional[ConsensusSettings] = None, **kwargs: Any) -> KLLMsChatCompletion:
        kwargs.pop("stream", None)
        settings = consensus_settings or ConsensusSettings()
        sampling = dict(temperature=temperature, max_tokens=max_tokens, top_p=top_p, frequency_penalty=frequency_penalty,
                        presence_penalty=presence_penalty, stop=stop, seed=seed, response_format=response_format)
        params = _call_params({"messages": messages, "model": model, "stream": False}, sampling, n, kwargs, settings)
        completion = await self._wrapper.client.chat.completions.create(**params)
        return await async_consolidate_chat_completions(completion, self._embed, client=self._wrapper.client, consensus_settings=settings)

    async def parse(self, *, messages: List[Any], model: str, response_format: Any, n: Optional[int] = None,
                    temperature: Optional[float] = None, max_tokens: Optional[int] = None, top_p: Optional[float] = None,
                    frequency_penalty: Optional[float] = None, presence_penalty: Optional[float] = None,
                    stop: Optional[Union[str, List[str]]] = None, seed: Optional[int] = None,
                    consensus_settings: Optional[ConsensusSettings] = None, **kwargs: Any) -> KLLMsParsedChatCompletion:
        settings = consensus_settings or ConsensusSettings()
        sampling = dict(temperature=temperature, max_tokens=max_tokens, top_p=top_p, frequency_penalty=frequency_penalty,
                        presence_penalty=presence_penalty, stop=stop, seed=seed)
        params = _call_params({"messages": messages, "model": model, "response_format": response_format}, sampling, n, kwargs, settings)
        completion = await self._wrapper.client.beta.chat.completions.parse(**params)
        return await async_consolidate_parsed_chat_completions(completion, self._embed, response_format=response_format,
                                                               client=self._wrapper.client, consensus_settings=settings)
