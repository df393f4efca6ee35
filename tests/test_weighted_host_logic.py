"""Likelihood-weighted consolidation without a GPU (self-defined semantics, DESIGN.md §5): the group-vote oracle against the C
oracle's K3b, the device JSON path's weighted phases instantiated on the host with the oracle in the kernels' place, and the
argument checks of the Python entry points and the client (stub OpenAI client, no network)."""
import ctypes as c
import json
import random

import numpy as np
import pytest

from k_llms_b200 import _native as K
from oracle import columnar as OC
from tests import weighted_oracle as W
from tests.helpers import jsongpu_with_oracle
from tests.test_gpu_json import _random_nested_record
from tests.test_jsongpu_host_logic import _flat_record, _shaped_record, s32_texts


def test_group_oracle_matches_k3b_oracle_on_regular_layouts():
    rng = np.random.default_rng(5)
    for n in (1, 2, 3, 5, 8, 17, 32, 33, 64):
        R, F = 20, 6
        codes = rng.integers(-2, 4, (R, F, n)).astype(np.int32)
        codes[:, 0, :] = rng.integers(0, 2, (R, n))  # some all-voting rows
        seq = (-rng.exponential(3.0, (R, n))).astype(np.float32)
        seq[: R // 2] = seq[: R // 2, :1]  # equal sums: weights exactly 1, integer class sums and ties
        _, emeta, _ = OC.weighted_vote(codes, seq)
        weight = np.stack([W.weights(s) for s in seq])
        meta, sums = W.vote_groups(codes.reshape(R * F, n), np.repeat(np.arange(R, dtype=np.int32), F), weight)
        assert np.array_equal(meta, emeta), n
        assert (sums[:, 1] >= sums[:, 0]).all()


def _naive_group(cells, w):
    """A second restatement: Counter-style tallies (dict of float32 sums), winner by sorted (-weight, first index)."""
    tally, first, count = {}, {}, {}
    wp = np.float32(0)
    for i, (cell, x) in enumerate(zip(cells, w)):
        if cell >= -1:
            wp = np.float32(wp + x)
        if cell >= 0:
            tally[cell] = np.float32(tally.get(cell, np.float32(0)) + x)
            first.setdefault(cell, i)
            count[cell] = count.get(cell, 0) + 1
    if not tally:
        return None, np.float32(0), wp, False
    best = sorted(tally, key=lambda k: (-tally[k], first[k]))[0]
    tie = sum(1 for k in tally if tally[k] == tally[best]) > 1
    return (first[best], count[best]), tally[best], wp, tie


def test_group_oracle_on_irregular_layouts():
    rng = random.Random(9)
    for _ in range(600):
        n = rng.choice([1, 2, 3, 5, 8, 16, 17, 32, 33, 64])
        n_rec = rng.randint(1, 4)
        spread = rng.choice([0.0, 1.0, 30.0, 200.0])  # 200: weights past the -87 clamp
        weight = np.stack([W.weights([np.float32(-rng.random() * spread) for _ in range(n)]) for _ in range(n_rec)])
        G = rng.randint(1, 6)
        cells = np.full((G, n), -2, dtype=np.int32)
        cand = np.zeros((G, n), dtype=np.int8)
        rec = np.array(sorted(rng.randrange(n_rec) for _ in range(G)), dtype=np.int32)
        for g in range(G):
            kept = sorted(rng.sample(range(n), rng.randint(1, n)))  # a dict / list filter keeps a subset, in order
            for i, k in enumerate(kept):
                cells[g, i] = rng.choice([-1, 0, 0, 1, 2, 3])
                cand[g, i] = k
        meta, sums = W.vote_groups(cells, rec, weight, cand)
        f = OC.meta_fields(meta)
        for g in range(G):
            w = [weight[rec[g]][cand[g, i]] if cells[g, i] >= -1 else np.float32(0) for i in range(n)]
            win, ww, wp, tie = _naive_group(cells[g], w)
            assert sums[g, 1] == wp and sums[g, 0] == ww
            assert f["present"][g] == int((cells[g] >= -1).sum()) and f["nn"][g] == int((cells[g] >= 0).sum())
            if win is None:
                assert f["flags"][g] == 0
            else:
                assert (f["idx"][g], f["support"][g]) == win and bool(f["flags"][g] & 4) == tie and f["flags"][g] & 1


def jsongpu_weighted_with_oracle(records, logprobs):
    """The weighted entry's phases on the host: kc_debug_jsongpu_plan -> K3 / weights / the weighted group vote by the oracle
    (vote records from kc_debug_jsongpu_vote_records) and the C oracle in K2 / K4's place -> kc_debug_jsongpu_emit_weighted."""
    lib = K.load()
    R = len(records)
    blob, off, n = K.pack_texts(records, pinned=False)
    h = c.c_void_p()
    K.check(lib.kc_debug_jsongpu_plan(blob.ctypes.data, off.ctypes.data, R, n, c.byref(h)))
    try:
        vc, nc, st = c.c_void_p(), c.c_void_p(), c.c_void_p()
        gv, gx = c.c_int64(), c.c_int64()
        K.check(lib.kc_debug_jsongpu_inputs(h, c.byref(vc), c.byref(gv), c.byref(nc), c.byref(gx), c.byref(st)))
        vmeta, vsums = np.zeros(max(gv.value, 1), dtype=np.uint32), np.zeros((max(gv.value, 1), 2), dtype=np.float32)
        nvalue, nmeta = np.zeros(max(gx.value, 1), dtype=np.float64), np.zeros(max(gx.value, 1), dtype=np.uint32)
        if gv.value:
            vr = c.c_void_p()
            K.check(lib.kc_debug_jsongpu_vote_records(h, c.byref(vr)))
            rec = np.ctypeslib.as_array(c.cast(vr, c.POINTER(c.c_int32)), shape=(gv.value,)).copy()
            codes = np.ctypeslib.as_array(c.cast(vc, c.POINTER(c.c_int8)), shape=(gv.value, n)).astype(np.int32)
            weight = np.stack([W.weights(W.seq_sums(lp)) for lp in logprobs])
            vmeta, vsums = W.vote_groups(codes, rec, weight)
        if gx.value:
            vals = np.ctypeslib.as_array(c.cast(nc, c.POINTER(c.c_double)), shape=(gx.value, n)).copy()
            nvalue, nmeta = OC.numeric(vals)
        mc, so, go, gm = c.c_void_p(), c.c_void_p(), c.c_void_p(), c.c_int64()
        K.check(lib.kc_debug_jsongpu_medoid_inputs(h, c.byref(mc), c.byref(so), c.byref(go), c.byref(gm)))
        midx, mavg = np.zeros(max(gm.value, 1), dtype=np.int32), np.zeros(max(gm.value, 1), dtype=np.float64)
        if gm.value:
            OC.lib().ko_medoid_str(mc, so, go, gm.value, midx.ctypes.data, mavg.ctypes.data)
        K.check(lib.kc_debug_jsongpu_set_medoid(h, midx.ctypes.data, mavg.ctypes.data))
        pc, po, pl, plo = c.c_void_p(), c.c_void_p(), c.c_void_p(), c.c_void_p()
        K.check(lib.kc_debug_jsongpu_emit_weighted(h, vmeta.ctypes.data, vsums.ctypes.data, nvalue.ctypes.data, nmeta.ctypes.data,
                                                   c.byref(pc), c.byref(po), c.byref(pl), c.byref(plo)))
        status = np.ctypeslib.as_array(c.cast(st, c.POINTER(c.c_uint8)), shape=(R,)).copy()
        co = np.ctypeslib.as_array(c.cast(po, c.POINTER(c.c_int64)), shape=(R + 1,))
        lo = np.ctypeslib.as_array(c.cast(plo, c.POINTER(c.c_int64)), shape=(R + 1,))
        return [None if status[r] else (c.string_at(pc.value + int(co[r]), int(co[r + 1] - co[r])).decode("ascii"),
                                         c.string_at(pl.value + int(lo[r]), int(lo[r + 1] - lo[r])).decode("ascii"))
                for r in range(R)]
    finally:
        lib.kc_debug_jsongpu_free(h)


def _records():
    rng = random.Random(77)
    out = {}
    for n in (2, 3, 5, 16, 33):
        out.setdefault(n, []).extend(s32_texts(12, n, 300 + n))
    for _ in range(300):
        n = rng.choice([2, 3, 4, 5, 8, 16])
        out.setdefault(n, []).append(_flat_record(rng, n))
    for _ in range(300):
        n = rng.choice([2, 3, 5, 8])
        out.setdefault(n, []).append(_shaped_record(rng, n))
    for _ in range(150):
        n = rng.choice([2, 3, 5])
        out.setdefault(n, []).append(_random_nested_record(rng, n))
    return out


def test_weighted_phases_equal_uniform_when_sums_are_equal():
    accepted = 0
    for n, recs in _records().items():
        uniform, _ = jsongpu_with_oracle(recs)
        weighted = jsongpu_weighted_with_oracle(recs, [W.equal_logprobs(n, k=1 + i % 40) for i in range(len(recs))])
        for u, w in zip(uniform, weighted):
            assert (u is None) == (w is None)
            accepted += u is not None
            assert u == w
    assert accepted > 600, accepted


def test_weighted_phases_match_the_weighted_oracle():
    from tests.helpers import raising_embeddings
    rng = random.Random(123)
    accepted = 0
    for n, recs in _records().items():
        lps = [W.random_logprobs(rng, n, scale=rng.choice([0.1, 1.0, 40.0])) for _ in recs]
        got = jsongpu_weighted_with_oracle(recs, lps)
        for texts, lp, g in zip(recs, lps, got):
            if g is None:
                continue
            accepted += 1
            content, lik = W.expected(texts, lp, embed=raising_embeddings)
            assert g == (content, lik), (texts, lp)
    assert accepted > 600, accepted


def test_weighting_changes_the_winner():
    """Three short, unlikely answers against two confident ones: uniform picks the three, likelihood the two."""
    texts = [json.dumps({"city": "Paris"})] * 2 + [json.dumps({"city": "Lyon"})] * 3
    lps = [[-0.01, -0.02]] * 2 + [[-3.0, -2.5]] * 3
    (u,), _ = jsongpu_with_oracle([texts])
    (w,) = jsongpu_weighted_with_oracle([texts], [lps])
    assert json.loads(u[0]) == {"city": "Lyon"} and json.loads(w[0]) == {"city": "Paris"}
    assert json.loads(w[1])["city"] > 0.9


# ----------------------------------------------------------------------------- argument checks (no device needed)


def test_value_errors():
    from k_llms_b200.utils.consensus_utils import ConsensusSettings, consensus_values, consensus_values_batch
    from k_llms_b200.utils.consolidation import consolidate_contents_batch
    lk = ConsensusSettings(candidate_weighting="likelihood")
    embed = lambda texts: [[0.0] for _ in texts]  # noqa: E731
    with pytest.raises(ValueError, match="logprobs"):
        consensus_values(["a", "b"], lk, embed, None)
    with pytest.raises(ValueError, match="2 candidates"):
        consensus_values(["a", "b"], lk, embed, None, candidate_logprobs=[[-1.0]])
    with pytest.raises(ValueError, match="NaN"):
        consensus_values(["a", "b"], lk, embed, None, candidate_logprobs=[[-1.0], [float("nan")]])
    with pytest.raises(ValueError, match="per record"):
        consensus_values_batch([["a", "b"]], lk, embed, candidate_logprobs=[])
    recs = [['{"a": 1}', '{"a": 2}']]
    with pytest.raises(ValueError, match="needs logprobs"):
        consolidate_contents_batch(recs, lk)
    with pytest.raises(ValueError, match="one sequence per candidate"):
        consolidate_contents_batch(recs, lk, logprobs=[[[-1.0]]])
    with pytest.raises(ValueError, match="NaN"):  # caught before any device work
        consolidate_contents_batch(recs, lk, logprobs=[[[-1.0], [float("nan")]]])
    assert ConsensusSettings().candidate_weighting == "uniform"
    with pytest.raises(Exception):
        ConsensusSettings(candidate_weighting="softmax")


def _completion(contents, logprobs):
    from openai.types.chat import ChatCompletion
    choices = []
    for i, (t, lp) in enumerate(zip(contents, logprobs)):
        ch = {"index": i, "finish_reason": "stop", "message": {"role": "assistant", "content": t}}
        if lp is not None:
            ch["logprobs"] = {"content": [{"token": "x", "logprob": x, "bytes": None, "top_logprobs": []} for x in lp]}
        choices.append(ch)
    return ChatCompletion.model_validate({"id": "x", "object": "chat.completion", "created": 0, "model": "m", "choices": choices})


class StubOpenAI:
    """Records the request and answers with a canned completion (no network)."""

    def __init__(self, completion):
        self.requests = []
        stub = self

        class _Completions:
            def create(self, **params):
                stub.requests.append(params)
                return completion

        class _Chat:
            completions = _Completions()

        self.chat = _Chat()


def test_missing_logprobs_on_a_kept_choice_raise():
    from k_llms_b200.utils.consensus_utils import ConsensusSettings
    from k_llms_b200.utils.consolidation import consolidate_chat_completions
    lk = ConsensusSettings(candidate_weighting="likelihood")
    comp = _completion(['{"a": "x"}', '{"a": "y"}', ""], [[-1.0], None, None])  # the empty choice is dropped, with its logprobs
    with pytest.raises(ValueError, match="candidate 1 has no logprobs"):
        consolidate_chat_completions(comp, lambda t: [[0.0] for _ in t], None, consensus_settings=lk)


def test_client_asks_for_logprobs_and_refuses_logprobs_false(monkeypatch):
    from types import SimpleNamespace

    from k_llms_b200.resources.completions import completions as CC
    from k_llms_b200.utils.consensus_utils import ConsensusSettings
    lk = ConsensusSettings(candidate_weighting="likelihood")
    comp = _completion(['{"a": "x"}', '{"a": "y"}'], [[-0.1], [-2.0]])
    seen = {}
    monkeypatch.setattr(CC, "consolidate_chat_completions",
                        lambda completion, embed, client, consensus_settings: seen.setdefault("settings", consensus_settings) or "ok")
    stub = StubOpenAI(comp)
    completions = CC.Completions(SimpleNamespace(client=stub))  # the wrapper's OpenAI client, stubbed
    completions.create(messages=[], model="m", n=2, consensus_settings=lk)
    assert stub.requests[-1]["logprobs"] is True and stub.requests[-1]["n"] == 2 and seen["settings"] is lk
    completions.create(messages=[], model="m", n=2)
    assert "logprobs" not in stub.requests[-1]
    with pytest.raises(ValueError, match="logprobs=False"):
        completions.create(messages=[], model="m", n=2, logprobs=False, consensus_settings=lk)
    assert len(stub.requests) == 2  # refused before the paid call
