"""CPU oracle of likelihood-weighted consolidation (self-defined semantics, DESIGN.md §5) — TEST INFRASTRUCTURE.

Restates, in plain Python + numpy float32, what the product computes with ConsensusSettings(candidate_weighting="likelihood"):

    sequence sums   K3's fixed-order fp32 sum of a candidate's token logprobs (the C oracle's ko_logprob_sum_f32)
    weights         w_c = kexp(s_c - max_k s_k) over a record's kept candidates (the C oracle's ko_exp_f32)
    group vote      kc_weighted_vote_groups_*: class weight = fp32 sum of its cells' weights in cell order, heaviest class wins,
                    equal weights -> the class whose first cell comes first; (W_win, W_present) with None cells in W_present
    object level    the dispatcher of oracle/consensus_py.py with the weights threaded through it: only str/bool vote leaves are
                    weighted, confidence round(pvf * (W_win / W_present), 5); numeric / medoid leaves are the unweighted oracle's
"""
from __future__ import annotations

import ctypes
import json
from typing import Callable, Optional, Sequence

import numpy as np

from oracle import columnar as OC
from oracle import consensus_py as O

F32 = np.float32
_exp = None


def kexp(x) -> np.float32:
    """ko_exp_f32 of the C oracle (bit-identical to the kernels' kexp)."""
    global _exp
    if _exp is None:
        _exp = OC.lib().ko_exp_f32
        _exp.argtypes = [ctypes.c_float]
        _exp.restype = ctypes.c_float
    return F32(_exp(float(F32(x))))


def seq_sums(token_logprobs: Sequence[Sequence[float]]) -> np.ndarray:
    """K3 over one sequence per candidate: float32 [n]."""
    lens = [len(s) for s in token_logprobs]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    flat = np.concatenate([np.asarray(s, dtype=np.float32) for s in token_logprobs] + [np.zeros(0, np.float32)])
    return OC.logprob_sum(flat if flat.size else np.zeros(1, np.float32), off)


def weights(sums) -> np.ndarray:
    """Candidate weights of one record from its kept candidates' sequence sums."""
    s = np.asarray(sums, dtype=np.float32)
    if s.size == 0:
        return s
    smax = s.max()
    return np.array([kexp(F32(x - smax)) for x in s], dtype=np.float32)


def group_vote(cells: Sequence[int], w: Sequence[np.float32]):
    """One group: cells in K1's coding (>= 0 class, -1 None, < -1 absent), w[i] = the weight of cell i's candidate.
    Returns (meta uint32, W_win float32, W_present float32)."""
    present = voters = 0
    w_present = F32(0.0)
    classes: dict = {}  # code -> [first cell, count, weight], first-seen order
    for i, c in enumerate(cells):
        if c < -1:
            continue
        present += 1
        w_present = F32(w_present + F32(w[i]))
        if c < 0:
            continue
        voters += 1
        if c not in classes:
            classes[c] = [i, 0, F32(0.0)]
        cl = classes[c]
        cl[1] += 1
        cl[2] = F32(cl[2] + F32(w[i]))
    if not voters:
        return _pack(0, 0, 0, present, 0), F32(0.0), w_present
    best = None
    for cl in classes.values():  # strict '>' in first-seen order: equal weights go to the class seen first
        if best is None or cl[2] > best[2]:
            best = cl
    tie = sum(1 for cl in classes.values() if cl[2] == best[2]) > 1
    return _pack(best[0], best[1], voters, present, 1 | (4 if tie else 0)), best[2], w_present


def _pack(idx, support, nn, present, flags) -> int:  # KC_META_PACK
    return (idx & 0x3F) | ((support & 0x7F) << 6) | ((nn & 0x7F) << 13) | ((present & 0x7F) << 20) | ((flags & 0x1F) << 27)


def vote_groups(cells: np.ndarray, rec: np.ndarray, weight: np.ndarray, cand: Optional[np.ndarray] = None):
    """kc_weighted_vote_groups_*: cells [G, n], rec int32 [G], weight float32 [R, n], cand int8 [G, n] or None ->
    (meta uint32 [G], sums float32 [G, 2])."""
    G, n = cells.shape
    meta = np.zeros(G, dtype=np.uint32)
    sums = np.zeros((G, 2), dtype=np.float32)
    for g in range(G):
        row = weight[rec[g]]
        w = [row[int(cand[g, i]) if cand is not None else i] if cells[g, i] >= -1 else F32(0.0) for i in range(n)]
        m, ww, wp = group_vote([int(x) for x in cells[g]], w)
        meta[g], sums[g, 0], sums[g, 1] = m, ww, wp
    return meta, sums


# ----------------------------------------------------------------------------- object level


def _vote(values, w, settings, pvf):
    """voting_consensus (oracle/consensus_py.py: vote) with candidate weights."""
    first = next((v for v in values if v is not None), None)
    if first is None:
        return None, pvf
    if isinstance(first, bool):
        keys = [v or False for v in values]
        cells, table = [], {}
        for k in keys:
            cells.append(table.setdefault(k, len(table)))
    else:
        keys, cells, table = [], [], {}
        for v in values:
            if v is None and not settings.allow_none_as_candidate:
                keys.append(None)
                cells.append(-1)
            else:
                k = None if v is None else O.sanitize(v)
                keys.append(k)
                cells.append(table.setdefault(k, len(table)))
    m, w_win, w_present = group_vote(cells, w)
    idx = m & 0x3F
    winner = keys[idx] if isinstance(first, bool) else values[idx]
    return winner, round(pvf * (float(w_win) / float(w_present)), 5)


def consensus(values: list, w: Sequence[np.float32], settings=O.DEFAULTS, pvf: float = 1.0, embed: Optional[Callable] = None):
    """oracle/consensus_py.py: consensus with w[c] = the weight of values[c]."""
    if not values:
        return None, pvf
    live = [v for v in values if v is not None]
    if not live:
        return None, 0.0
    head = live[0]
    if isinstance(head, (str, bool)) and all(len(str(v).strip().split()) < 3 for v in live):
        return _vote(values, w, settings, pvf)
    if isinstance(head, dict):
        kept = [(v, x) for v, x in zip(values, w) if isinstance(v, dict)]
        dicts, dw = [v for v, _ in kept], [x for _, x in kept]
        sub = pvf * (len(dicts) / len(values))
        keys: dict = {}
        for d in dicts:
            for k in d:
                keys.setdefault(k, None)
        out, conf = {}, {}
        for k in keys:
            if any(mk in k for mk in O.SKIPPED_KEY_MARKERS):
                continue
            out[k], conf[k] = consensus([d.get(k) for d in dicts], dw, settings, sub, embed)
        return out, conf
    if isinstance(head, list):
        kept = [(v, x) for v, x in zip(values, w) if isinstance(v, list)]
        lists, lw = [v for v, _ in kept], [x for _, x in kept]
        sub = pvf * (len(lists) / len(values))
        longest = max(len(l) for l in lists)
        if longest == 0:
            return [], []
        pairs = [consensus([l[i] if i < len(l) else None for l in lists], lw, settings, sub, embed) for i in range(longest)]
        return [p[0] for p in pairs], [p[1] for p in pairs]
    sub = pvf * (len(live) / len(values))
    return O.primitive(live, settings, sub, embed)


def client_order(values: list, token_logprobs: Sequence[Sequence[float]], settings=O.DEFAULTS, embed: Optional[Callable] = None):
    """O.client_order with likelihood weighting: values = the kept contents, token_logprobs[c] = candidate c's logprobs."""
    w = weights(seq_sums(token_logprobs))
    aligned = [(d if isinstance(d, dict) else {}) for d in O.align_flat(values)] if len(values) >= 2 else values
    return consensus(aligned, w, settings, 1.0, embed)


def expected(texts: Sequence[str], token_logprobs: Sequence[Sequence[float]], embed: Optional[Callable] = None, aligned=None):
    """(consensus content text, likelihoods text) of one record as consolidate_contents_batch(..., logprobs=...) returns them
    (likelihoods as JSON text).  aligned: the record's contents after the list alignment pre-pass, when it has lists."""
    from k_llms_b200.utils.consolidation import _format_consensus_content, _safe_parse_content
    kept = [(t, lp) for t, lp in zip(texts, token_logprobs) if t]
    contents = [_safe_parse_content(t) for t, _ in kept]
    lps = [lp for _, lp in kept]
    if aligned is not None:
        value, conf = consensus([(d if isinstance(d, dict) else {}) for d in aligned], weights(seq_sums(lps)), O.DEFAULTS, 1.0, embed)
    else:
        value, conf = client_order(contents, lps, embed=embed)
    return _format_consensus_content(value), json.dumps(conf)


def random_logprobs(rng, n_cand: int, lo: int = 0, hi: int = 12, scale: float = 1.0):
    """n_cand sequences of lo..hi token logprobs (float32-representable, <= 0)."""
    return [[float(F32(-rng.expovariate(1.0) * scale)) for _ in range(rng.randint(lo, hi))] for _ in range(n_cand)]


def equal_logprobs(n_cand: int, k: int = 5, v: float = -0.25):
    """n_cand identical sequences: every sequence sum is the same, every weight exactly 1.0f."""
    return [[v] * k for _ in range(n_cand)]
