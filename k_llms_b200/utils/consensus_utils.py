"""Drop-in for `k_llms.utils.consensus_utils` — the seven names `consolidation.py` imports
(reference consolidation.py:11-19) — with the scalar-field consensus on the GPU.

`consensus_values` keeps the reference signature and return shape (consensus_utils.py:1376-1382, "cu"):
the recursion over dicts and lists is planned on the host (k_llms_b200.columnar), every str/bool vote
(cu:936-982) and every numeric clustering (cu:1098-1219) of the record runs in ONE launch each of the sm_100a
kernels behind `libkllms_b200.so`, and the result tree is rebuilt.  `consensus_values_batch` is the new batched
entry (many records per launch) the reference lacks.

There is NO CPU implementation of the hot path here: without the CUDA library or a device these functions raise.
"""
from __future__ import annotations

import asyncio
import logging
import math
import warnings
from typing import Any, Awaitable, Callable, List, Literal, Optional, Sequence, Tuple

from pydantic import BaseModel

from .. import columnar
from . import similarity

logger = logging.getLogger(__name__)

StringSimilarityMethod = Literal["levenshtein", "jaccard", "hamming", "embeddings"]
StringConsensusMethod = Literal["centroid", "llm-consensus"]
CandidateWeighting = Literal["uniform", "likelihood"]
SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE = Callable[[List[str]], List[List[float]]]
ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE = Callable[[List[str]], Awaitable[List[List[float]]]]


class ConsensusSettings(BaseModel):
    """Same fields and defaults as the reference model (cu:53-69).  Only allow_none_as_candidate,
    string_similarity_method, string_consensus_method, min_support_ratio, rel_eps and abs_eps are read by
    the reference's code paths; the others are accepted for compatibility.

    candidate_weighting is this package's own (self-defined, DESIGN.md §5): "uniform" (default) is the reference's vote;
    "likelihood" weights every candidate's vote in str/bool fields by exp(s_c - max_k s_k), s_c = the sum of the candidate's
    token logprobs.  Numeric fields, similarity-medoid fields and the list alignment are not weighted."""

    allow_none_as_candidate: bool = False
    string_similarity_method: StringSimilarityMethod = "embeddings"
    string_consensus_method: StringConsensusMethod = "centroid"
    minimum_voters_threshold: float = 0.75
    min_support_ratio: float = 0.51
    rel_eps: float = 0.03
    abs_eps: float = 1e-6
    base_maj_thresh: float = 0.6
    maj_loosen_k: float = 0.1
    trim_frac: float = 0.2
    candidate_weighting: CandidateWeighting = "uniform"


def check_candidate_logprobs(settings: ConsensusSettings, candidate_logprobs, n: int):
    """The logprobs a likelihood-weighted consolidation runs on: candidate_logprobs[c] = the token logprobs of candidate c (one
    sequence per candidate), as lists of floats; None under uniform weighting.  Raises ValueError when they are missing, do not
    match the n candidates, or hold a NaN."""
    if settings.candidate_weighting != "likelihood":
        return None
    if candidate_logprobs is None:
        raise ValueError("candidate_weighting='likelihood' needs the token logprobs of every candidate (request logprobs=True)")
    if len(candidate_logprobs) != n:
        raise ValueError(f"candidate_weighting='likelihood': {len(candidate_logprobs)} logprob sequences for {n} candidates")
    out = []
    for c, seq in enumerate(candidate_logprobs):
        if seq is None:
            raise ValueError(f"candidate_weighting='likelihood': candidate {c} has no logprobs (request logprobs=True)")
        seq = [float(x) for x in seq]
        if any(math.isnan(x) for x in seq):
            raise ValueError(f"candidate_weighting='likelihood': candidate {c} has a NaN logprob")
        out.append(seq)
    return out


def _host_primitive(settings: ConsensusSettings):
    def run(values: list, parent_valid_frac: float, embed):
        if isinstance(values[0], str) and settings.string_consensus_method == "llm-consensus" \
                and settings.string_similarity_method == "embeddings":
            # cu:1090-1096 asks gpt-5-mini for a consensus string: a network call, outside this build's scope
            raise NotImplementedError("string_consensus_method='llm-consensus' needs a network LLM call; use 'centroid'")
        return similarity.medoid(values, settings.string_similarity_method, embed, parent_valid_frac)
    return run


def _plan_for(n: int, settings: ConsensusSettings, numeric_branch: bool = True) -> columnar.Plan:
    plan = columnar.Plan(n, settings.allow_none_as_candidate, settings.rel_eps, settings.abs_eps, _host_primitive(settings),
                         numeric_branch=numeric_branch, weighted=settings.candidate_weighting == "likelihood")
    plan.string_method = settings.string_similarity_method if settings.string_consensus_method == "centroid" else "host"
    return plan


def consensus_values(
    values: List[Any],
    consensus_settings: ConsensusSettings,
    sync_get_openai_embeddings_from_text: SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    parent_valid_frac: float = 1.0,
    _numeric_branch: bool = True,
    *,
    candidate_logprobs: Optional[Sequence[Sequence[float]]] = None,
) -> Tuple[Any, Any]:
    """(consensus value, confidence) for one record's n candidate values — cu:1376-1454.  With
    consensus_settings.candidate_weighting == "likelihood", candidate_logprobs[c] = the token logprobs of values[c]."""
    lps = check_candidate_logprobs(consensus_settings, candidate_logprobs, len(values))
    plan = _plan_for(len(values), consensus_settings, _numeric_branch)
    root = plan.add(values, parent_valid_frac, sync_get_openai_embeddings_from_text, lps)
    res = plan.run() if (plan.vote_rows or plan.num_rows or plan.medoid_groups) else {}
    return plan.materialise(root, res)


def consensus_values_batch(
    records: Sequence[List[Any]],
    consensus_settings: Optional[ConsensusSettings] = None,
    sync_get_openai_embeddings_from_text: Optional[SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE] = None,
    client: Any = None,
    parent_valid_frac: float = 1.0,
    *,
    candidate_logprobs: Optional[Sequence[Sequence[Sequence[float]]]] = None,
) -> List[Tuple[Any, Any]]:
    """Batched entry (new): consensus_values for many independent records with ONE K1 and ONE K2 launch.  With likelihood
    weighting, candidate_logprobs[r][c] = the token logprobs of records[r][c]."""
    settings = consensus_settings or ConsensusSettings()
    embed = sync_get_openai_embeddings_from_text if sync_get_openai_embeddings_from_text is not None else _no_embeddings
    if settings.candidate_weighting == "likelihood" and (candidate_logprobs is None or len(candidate_logprobs) != len(records)):
        raise ValueError("candidate_weighting='likelihood' needs one list of candidate logprobs per record")
    lps = [check_candidate_logprobs(settings, candidate_logprobs[i] if candidate_logprobs is not None else None, len(values))
           for i, values in enumerate(records)]
    plan = _plan_for(max((len(r) for r in records), default=1), settings)
    roots = [plan.add(values, parent_valid_frac, embed, lp) for values, lp in zip(records, lps)]
    res = plan.run() if (plan.vote_rows or plan.num_rows or plan.medoid_groups) else {}
    return [plan.materialise(root, res) for root in roots]


def _no_embeddings(texts):
    raise RuntimeError("no embeddings callable was supplied")  # the similarity code then falls back to Levenshtein


async def async_consensus_values(
    values: List[Any],
    consensus_settings: ConsensusSettings,
    async_get_openai_embeddings_from_text: ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    parent_valid_frac: float = 1.0,
    *,
    candidate_logprobs: Optional[Sequence[Sequence[float]]] = None,
) -> Tuple[Any, Any]:
    """Async twin (cu:1779-1860).  The reference's async primitive has NO numeric clustering (cu:1638-1688, SURVEY.md §0.5):
    a non-unanimous numeric field takes the similarity medoid — [10, 10, 11] gives (10, 0.5) here and (10.0, 0.66667) in the
    sync path.  That difference is part of the reference's behaviour and is reproduced; votes still run on the GPU, off the
    event loop."""
    loop = asyncio.get_running_loop()

    def embed(texts):
        fut = asyncio.run_coroutine_threadsafe(async_get_openai_embeddings_from_text(texts), loop)
        return fut.result()

    return await asyncio.to_thread(consensus_values, values, consensus_settings,
                                   embed if async_get_openai_embeddings_from_text is not None else None, client,
                                   parent_valid_frac, False, candidate_logprobs=candidate_logprobs)


# ----------------------------------------------------------------------------- alignment pre-pass


def recursive_list_alignments(
    values: List[Any],
    string_similarity_method: StringSimilarityMethod,
    sync_get_openai_embeddings_from_text: SYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    min_support_ratio: float,
    max_novelty_ratio: float = 0.25,
    current_path: str = "",
    reference_idx: Optional[int] = None,
):
    """The pre-pass `consolidation.py` runs before the vote (cu:458-613).

    Dict payloads: every candidate gets every key, keys sorted, missing -> None, recursively (cu:516-548) — this is
    what flat records need and it is implemented here.  Lists are aligned by the separate module
    `k_llms_b200.utils.list_alignment` (reference cu:185-430 + majority_sorting.py)."""
    from copy import deepcopy
    if not values:
        return values, {}
    if all(v is None for v in values):
        return values, {current_path: [current_path for _ in values]}
    non_nulls = [v for v in values if v is not None]
    values = deepcopy(values)  # cu:504
    first_type = type(non_nulls[0])
    same_type = all(isinstance(x, first_type) for x in non_nulls)
    key_mappings: dict = {}
    if not same_type or first_type not in (dict, list):
        key_mappings[current_path] = [current_path if (v is not None or idx == reference_idx) else None
                                      for idx, v in enumerate(values)]
        return values, key_mappings
    if first_type is dict:
        dicts_only = [(d if isinstance(d, dict) else {}) for d in values]
        all_keys = sorted({k for d in dicts_only for k in d})
        for key in all_keys:
            sub_path = f"{current_path}.{key}" if current_path else key
            aligned, sub_map = recursive_list_alignments(
                [d.get(key) for d in dicts_only], string_similarity_method, sync_get_openai_embeddings_from_text, client,
                min_support_ratio, max_novelty_ratio=max_novelty_ratio, current_path=sub_path, reference_idx=reference_idx)
            for d, v in zip(dicts_only, aligned):
                d[key] = v
            key_mappings.update(sub_map)
        return [{k: d.get(k) for k in all_keys} for d in dicts_only], key_mappings
    from .list_alignment import align_list_values
    return align_list_values(values, string_similarity_method, sync_get_openai_embeddings_from_text, client, min_support_ratio,
                             max_novelty_ratio, current_path, reference_idx, recursive_list_alignments)


async def async_recursive_list_alignments(
    values: List[Any],
    string_similarity_method: StringSimilarityMethod,
    async_get_openai_embeddings_from_text: ASYNC_GET_OPENAI_EMBEDDINGS_FROM_TEXT_TYPE,
    client: Any,
    min_support_ratio: float,
    max_novelty_ratio: float = 0.25,
    current_path: str = "",
    reference_idx: Optional[int] = None,
):
    loop = asyncio.get_running_loop()

    def embed(texts):
        return asyncio.run_coroutine_threadsafe(async_get_openai_embeddings_from_text(texts), loop).result()

    return await asyncio.to_thread(recursive_list_alignments, values, string_similarity_method, embed, client,
                                   min_support_ratio, max_novelty_ratio, current_path, reference_idx)
