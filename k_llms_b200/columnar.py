"""Host prologue / epilogue of the CUDA consensus path: flatten candidate objects into columnar groups,
run K1/K2 once over ALL groups of ALL records, rebuild the (value, confidence) trees.

The recursion mirrors the reference dispatcher `consensus_values` (consensus_utils.py:1376-1454, "cu") but
instead of computing a scalar field it RECORDS it as a group:

  * vote group    (cu:1405-1411 -> voting_consensus cu:936-982): cells = local dictionary codes of the
    processed values (`sanitize_value(v)` cu:925-933 for strings, `v or False` cu:956 for bools), None = -1
  * numeric group (cu:1443-1453 -> consensus_as_primitive cu:1098-1219): cells = float(v); None, bools,
    strings, nan/inf are tagged so the kernel counts them exactly as the reference does (cu:1100-1114)

The shape of the result (dict keys in first-seen order cu:1281-1282, list lengths cu:1332-1341, the
parent_valid_frac products cu:1418,1433,1444) depends only on the input structure, so it is fixed while
planning; the GPU fills in the leaves.  Multi-word string fields (the similarity medoid, cu:1221-1237) are recorded as
medoid groups for K4 when every pair is a Levenshtein pair inside the kernel's contract (`Plan._medoid_on_device`);
mixed payloads and the other similarity methods are computed by `k_llms_b200.utils.similarity` on the host.

With `weighted=True` (ConsensusSettings.candidate_weighting == "likelihood", self-defined: DESIGN.md §5) every record comes with
its candidates' token logprobs; each vote group also records the record and, per cell, the ORIGINAL candidate index of the value
(consensus_dict / consensus_list keep only the candidates whose value is a dict / list, cu:1416,1431, so positions shift), and the
vote groups are decided by K3 -> candidate weights -> kc_weighted_vote_groups_i32 instead of K1.  Numeric and medoid leaves are
not weighted.
"""
from __future__ import annotations

import math
import re
from typing import Any, Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native

MAX_CANDIDATES = _native.MAX_CANDIDATES
SKIPPED_KEY_MARKERS = ("reasoning___", "source___")  # cu:1287

_F64_NONE = np.array([_native.F64_NONE_BITS], dtype=np.uint64).view(np.float64)[0]
_F64_ABSENT = np.array([_native.F64_ABSENT_BITS], dtype=np.uint64).view(np.float64)[0]


# ----------------------------------------------------------------------------- sanitising (cu:925-933)

try:  # a dependency of the package (pyproject.toml), as of the reference (requirements.txt); ASCII input never reaches it
    from unidecode import unidecode as _unidecode  # type: ignore
except Exception:  # pragma: no cover - depends on the image
    _unidecode = None


def _fold_non_ascii(s: str) -> str:
    """unidecode(s) (cu:931).  Without the Unidecode package the vote classes of non-ASCII text would differ from the
    reference's ('Straße' / 'Strasse' share a class under unidecode), so this fails loudly instead of guessing — unless
    KLLMS_B200_ALLOW_NFKD=1 opts into NFKD folding (a documented deviation: combining marks are dropped, ß ø æ CJK are not
    transliterated)."""
    if _unidecode is not None:
        return _unidecode(s)
    import os
    if os.environ.get("KLLMS_B200_ALLOW_NFKD") != "1":
        raise ImportError("non-ASCII text needs the Unidecode package (a dependency of k_llms_b200, see pyproject.toml) to be "
                          "sanitised like the reference does; install it, or set KLLMS_B200_ALLOW_NFKD=1 to accept NFKD folding")
    import unicodedata
    return "".join(ch for ch in unicodedata.normalize("NFKD", s) if not unicodedata.combining(ch))


def _normalize(text: str) -> str:
    """normalize_string (cu:660-673): keep ASCII alphanumerics, lower-case."""
    return "".join(ch for ch in text if ch.isascii() and ch.isalnum()).lower() if text else ""


_NOT_ALNUM = re.compile(r"[^a-zA-Z0-9]")


def sanitize_value(v: Any) -> str:
    """str() -> lower -> drop spaces -> unidecode -> keep [a-zA-Z0-9]  (cu:925-933)."""
    s = str(v).lower().replace(" ", "")
    if not s.isascii():
        s = _fold_non_ascii(s)
    return _NOT_ALNUM.sub("", s)


# ----------------------------------------------------------------------------- plan nodes


class _Const:
    __slots__ = ("value", "conf")

    def __init__(self, value, conf):
        self.value, self.conf = value, conf


class _VoteLeaf:
    __slots__ = ("row", "cells", "pvf")

    def __init__(self, row: int, cells: list, pvf: float):
        self.row, self.cells, self.pvf = row, cells, pvf  # cells[i] = value returned when cell i wins


class _NumLeaf:
    __slots__ = ("row", "cells", "pvf")

    def __init__(self, row: int, cells: list, pvf: float):
        self.row, self.cells, self.pvf = row, cells, pvf


class _MedoidLeaf:
    __slots__ = ("row", "cells", "pvf")

    def __init__(self, row: int, cells: list, pvf: float):
        self.row, self.cells, self.pvf = row, cells, pvf


class _DictNode:
    __slots__ = ("children",)

    def __init__(self, children: dict):
        self.children = children


class _ListNode:
    __slots__ = ("children",)

    def __init__(self, children: list):
        self.children = children


class Plan:
    """Leaf groups of one or many records, ready for one K1, one K2 and one K4 launch."""

    def __init__(self, n: int, allow_none_as_candidate: bool, rel_eps: float, abs_eps: float, host_primitive: Callable,
                 numeric_branch: bool = True, weighted: bool = False):
        if n > MAX_CANDIDATES:
            raise ValueError(f"{n} candidates per request: k_llms_b200 consolidates at most {MAX_CANDIDATES} (one kernel row per "
                             "field holds every candidate; the package has no CPU path to fall back to)")
        # False: the reference's ASYNC dispatcher, whose primitive has no numeric clustering (cu:1638-1688): numbers take the
        # similarity medoid like any other non-enum value
        self.numeric_branch = numeric_branch
        self.n = max(n, 1)
        self.allow_none = allow_none_as_candidate
        self.rel_eps, self.abs_eps = rel_eps, abs_eps
        self.host_primitive = host_primitive
        self.vote_rows: List[List[int]] = []
        self.num_rows: List[List[float]] = []
        self.medoid_groups: List[List[str]] = []  # normalised strings of the groups K4 handles
        self.string_method = "embeddings"         # set by the caller (ConsensusSettings.string_similarity_method)
        self.weighted = weighted
        self.rec_logprobs: List[Sequence[Sequence[float]]] = []  # weighted: per record, the token logprobs of each candidate
        self.vote_rec: List[int] = []             # weighted: the record of each vote row
        self.vote_cand: List[List[int]] = []      # weighted: the candidate of each cell of each vote row
        self._rec = -1

    # -- leaves ---------------------------------------------------------------------------------------
    def _vote(self, values: Sequence[Any], pvf: float, cand: Sequence[int]) -> _VoteLeaf:
        first = next(v for v in values if v is not None)
        codes: List[int] = []
        table: dict = {}
        if isinstance(first, bool):  # cu:954-958: None and every falsy value become False
            cells = [v or False for v in values]
            for k in cells:
                codes.append(table.setdefault(k, len(table)))
        else:
            cells = list(values)
            for v in values:
                if v is None and not self.allow_none:
                    codes.append(_native.CODE_NONE)  # cu:964: None does not vote
                else:
                    k = None if v is None else sanitize_value(v)
                    codes.append(table.setdefault(k, len(table)))
        codes.extend([_native.CODE_ABSENT] * (self.n - len(codes)))
        self.vote_rows.append(codes)
        if self.weighted:
            self.vote_rec.append(self._rec)
            self.vote_cand.append(list(cand) + [0] * (self.n - len(cand)))
        return _VoteLeaf(len(self.vote_rows) - 1, cells, pvf)

    def _numeric(self, values: Sequence[Any], pvf: float) -> _NumLeaf:
        row: List[float] = []
        for v in values:
            if v is None:
                row.append(_F64_NONE)
            elif isinstance(v, bool) or not isinstance(v, (int, float)):
                row.append(math.nan)  # present, counted in `total`, never clustered (cu:1106-1108)
            else:
                try:
                    row.append(float(v))  # non-finite floats are dropped by the kernel (cu:1111)
                except OverflowError:
                    row.append(math.nan)  # cu:1113-1114
        row.extend([_F64_ABSENT] * (self.n - len(row)))
        self.num_rows.append(row)
        return _NumLeaf(len(self.num_rows) - 1, list(values), pvf)

    # -- dispatcher (cu:1376-1454) ----------------------------------------------------------------------
    def add(self, values: Sequence[Any], pvf: float, embed: Optional[Callable],
            candidate_logprobs: Optional[Sequence[Sequence[float]]] = None):
        """Plan one record; a weighted plan needs candidate_logprobs[c] = the token logprobs of values[c]."""
        if self.weighted:
            if candidate_logprobs is None or len(candidate_logprobs) != len(values):
                raise ValueError("a likelihood-weighted plan needs the token logprobs of every candidate")
            self.rec_logprobs.append(candidate_logprobs)
            self._rec = len(self.rec_logprobs) - 1
        return self._add(values, pvf, embed, range(len(values)))

    def _add(self, values: Sequence[Any], pvf: float, embed: Optional[Callable], cand: Sequence[int]):
        if not values:
            return _Const(None, pvf)  # cu:1395-1396
        live = [v for v in values if v is not None]
        if not live:
            return _Const(None, 0.0)  # cu:1401-1402
        head = live[0]
        if isinstance(head, (str, bool)) and all(len(str(v).strip().split()) < 3 for v in live):
            return self._vote(values, pvf, cand)  # cu:1405-1411
        if isinstance(head, dict):  # cu:1414-1426 -> consensus_dict cu:1269-1306
            kept = [(c, v) for c, v in zip(cand, values) if isinstance(v, dict)]
            dicts, sub_cand = [v for _, v in kept], [c for c, _ in kept]
            sub = pvf * (len(dicts) / len(values))
            keys: dict = {}
            for d in dicts:
                for k in d:
                    keys.setdefault(k, None)
            children = {}
            for k in keys:
                if any(mark in k for mark in SKIPPED_KEY_MARKERS):
                    continue
                children[k] = self._add([d.get(k) for d in dicts], sub, embed, sub_cand)
            return _DictNode(children)
        if isinstance(head, list):  # cu:1429-1441 -> consensus_list cu:1309-1352
            kept = [(c, v) for c, v in zip(cand, values) if isinstance(v, list)]
            lists, sub_cand = [v for _, v in kept], [c for c, _ in kept]
            sub = pvf * (len(lists) / len(values))
            longest = max(len(l) for l in lists)
            return _ListNode([self._add([l[i] if i < len(l) else None for l in lists], sub, embed, sub_cand) for i in range(longest)])
        if embed is None:  # cu:1445-1446
            raise ValueError("sync_get_openai_embeddings_from_text is required for primitive consensus")
        try:
            numeric_like = isinstance(type(head)(), (int, float))  # cu:1099
        except Exception:
            numeric_like = False
        if self.numeric_branch and (numeric_like or all(isinstance(v, (int, float)) for v in live)):
            # the kernel applies the None-stripping and len(values) bookkeeping of cu:1444 / cu:1082-1086 itself
            return self._numeric(values, pvf)
        sub = pvf * (len(live) / len(values))  # cu:1444
        if len(live) == 1:
            return _Const(live[0], sub * (1 / 1))  # cu:1085-1086
        if self._medoid_on_device(live):
            self.medoid_groups.append([_normalize(s) for s in live])
            return _MedoidLeaf(len(self.medoid_groups) - 1, live, sub)
        value, conf = self.host_primitive(live, sub, embed)  # similarity medoid on the host, cu:1221-1237
        return _Const(value, conf)

    def _medoid_on_device(self, live: Sequence[Any]) -> bool:
        """K4 takes groups of plain ASCII strings: methods 'jaccard' and 'hamming' always; 'levenshtein' when every pair has a
        <= 64-character side; 'embeddings' where, further, no two strings are both longer than 50 characters (cu:813 would ask
        the embeddings service for those)."""
        if self.string_method not in ("levenshtein", "embeddings", "jaccard", "hamming") or len(live) > MAX_CANDIDATES:
            return False
        if not all(isinstance(v, str) and v.isascii() for v in live):
            return False
        if self.string_method == "embeddings" and sum(1 for v in live if len(v) > 50) > 1:
            return False
        lens = [len(_normalize(v)) for v in live]
        if self.string_method in ("jaccard", "hamming"):  # character sets / position-wise mismatches: no pattern-length contract
            return max(lens) <= 2000
        return sum(1 for l in lens if l > 64) <= 1 and max(lens) <= 2000

    # -- device ----------------------------------------------------------------------------------------
    def run(self, device=None):
        """One K1, one K2 and one K4 launch over every recorded group; returns numpy result columns."""
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("k_llms_b200: no CUDA device — the consensus hot path has no CPU fallback")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        out = {}
        if self.vote_rows and self.weighted:
            codes = torch.from_numpy(np.asarray(self.vote_rows, dtype=np.int32)).to(dev)
            meta, sums = _native.weighted_vote_groups(codes, torch.tensor(self.vote_rec, dtype=torch.int32, device=dev),
                                                      self._candidate_weights(torch, dev),
                                                      torch.from_numpy(np.asarray(self.vote_cand, dtype=np.int8)).to(dev))
            out["vote_meta"] = meta.cpu().numpy().view(np.uint32)
            out["vote_sums"] = sums.cpu().numpy()
        elif self.vote_rows:
            codes = torch.from_numpy(np.asarray(self.vote_rows, dtype=np.int32)).to(dev)
            _, meta = _native.vote(codes, None)
            out["vote_meta"] = meta.cpu().numpy().view(np.uint32)
        if self.num_rows:
            vals = torch.from_numpy(np.asarray(self.num_rows, dtype=np.float64)).to(dev)
            value, meta = _native.numeric(vals, self.rel_eps, self.abs_eps)
            out["num_value"] = value.cpu().numpy()
            out["num_meta"] = meta.cpu().numpy().view(np.uint32)
        if self.medoid_groups:
            blobs, str_off, grp_off = [], [0], [0]
            for grp in self.medoid_groups:
                for s in grp:
                    b = s.encode("ascii")
                    blobs.append(b)
                    str_off.append(str_off[-1] + len(b))
                grp_off.append(grp_off[-1] + len(grp))
            chars = np.frombuffer(b"".join(blobs) or b"\0", dtype=np.uint8).copy()
            idx, avg = _native.medoid_str(torch.from_numpy(chars).to(dev), torch.tensor(str_off, dtype=torch.int32, device=dev),
                                          torch.tensor(grp_off, dtype=torch.int32, device=dev),
                                          max_group=max(len(grp) for grp in self.medoid_groups), method=self.string_method)
            out["medoid_idx"], out["medoid_avg"] = idx.cpu().numpy(), avg.cpu().numpy()
        return out

    def _candidate_weights(self, torch, dev):
        """K3 over every candidate's token logprobs, then the weight pre-pass: float32 [records, n].  A record with fewer than n
        candidates fills the rest of its row with -3.0e38 (never the record's maximum, never referenced by a cell)."""
        seqs = [s for rec in self.rec_logprobs for s in rec]
        slots = [r * self.n + c for r, rec in enumerate(self.rec_logprobs) for c in range(len(rec))]
        lens = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
        offsets = np.zeros(len(seqs) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        flat = np.zeros(max(int(offsets[-1]), 1), dtype=np.float32)
        if offsets[-1]:
            flat[:offsets[-1]] = np.concatenate([np.asarray(s, dtype=np.float32) for s in seqs if len(s)])
        sums = _native.logprob_sum(torch.from_numpy(flat).to(dev), torch.from_numpy(offsets).to(dev))
        seq = torch.full((len(self.rec_logprobs) * self.n,), -3.0e38, dtype=torch.float32, device=dev)
        seq[torch.tensor(slots, dtype=torch.int64, device=dev)] = sums
        return _native.candidate_weights(seq.view(len(self.rec_logprobs), self.n))

    # -- epilogue --------------------------------------------------------------------------------------
    @staticmethod
    def _fields(m: int) -> Tuple[int, int, int, int, int]:
        return m & 0x3F, (m >> 6) & 0x7F, (m >> 13) & 0x7F, (m >> 20) & 0x7F, (m >> 27) & 0x1F

    def materialise(self, node, res) -> Tuple[Any, Any]:
        if isinstance(node, _Const):
            return node.value, node.conf
        if isinstance(node, _DictNode):
            val, conf = {}, {}
            for k, child in node.children.items():
                val[k], conf[k] = self.materialise(child, res)
            return val, conf
        if isinstance(node, _ListNode):
            pairs = [self.materialise(c, res) for c in node.children]
            return [p[0] for p in pairs], [p[1] for p in pairs]
        if isinstance(node, _MedoidLeaf):  # cu:1233-1237
            return node.cells[int(res["medoid_idx"][node.row])], round(node.pvf * float(res["medoid_avg"][node.row]), 5)
        if isinstance(node, _VoteLeaf):
            idx, support, _nn, present, flags = self._fields(int(res["vote_meta"][node.row]))
            if not flags & _native.FLAG_HAS_VALUE:  # cannot happen for a planned vote group (>= 1 voter)
                return None, (node.pvf if present == 0 else 0.0)
            if "vote_sums" in res:  # likelihood-weighted: the weighted form of support / present (DESIGN.md §5)
                w_win, w_present = res["vote_sums"][node.row]
                return node.cells[idx], round(node.pvf * (float(w_win) / float(w_present)), 5)
            return node.cells[idx], round(node.pvf * (support / present), 5)  # cu:971,973,982
        idx, support, nn, present, flags = self._fields(int(res["num_meta"][node.row]))
        if flags & _native.FLAG_HAS_VALUE:
            if flags & _native.FLAG_SINGLE:
                return node.cells[idx], node.pvf * (1 / present) * (1 / 1)  # cu:1444, cu:1085-1086
            return float(res["num_value"][node.row]), round(support / nn, 5)  # cu:1176-1178,1217-1219
        if flags & _native.FLAG_NO_FINITE:
            return None, node.pvf * (nn / present)  # cu:1444, cu:1115-1116
        return None, (node.pvf if present == 0 else 0.0)
