"""Likelihood-weighted consolidation on the B200 (self-defined semantics, DESIGN.md §5): the weight pre-pass and both group-vote
kernels bit for bit against the oracle, consolidate_contents_batch(..., logprobs=...) on the device path and the Python path, a
config-4-shaped batch through the weighted device JSON entry, and the client with a stub OpenAI client."""
import json
import random

import numpy as np
import pytest

from tests import weighted_oracle as W
from tests.helpers import raising_embeddings

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 16, 17, 32, 33, 64])
def test_group_kernels_match_the_oracle(torch, n):
    from k_llms_b200 import _native as K
    rng = random.Random(1000 + n)
    R = 300
    seq = np.full((R, n), -3.0e38, dtype=np.float32)
    n_kept = []
    for r in range(R):
        k = rng.randint(1, n)  # a record may keep fewer candidates than the batch's n
        spread = rng.choice([0.0, 0.5, 20.0, 300.0])  # 300: weights past the -87 clamp
        seq[r, :k] = [np.float32(-rng.random() * spread) for _ in range(k)]
        n_kept.append(k)
    weight = K.candidate_weights(torch.from_numpy(seq).cuda()).cpu().numpy()
    for r in range(R):
        ew = W.weights(seq[r, :n_kept[r]])
        assert np.array_equal(weight[r, :n_kept[r]].view(np.uint32), ew.view(np.uint32)), r
    cells, rec, cand = [], [], []
    for r in range(R):  # ragged groups per record, contiguous per record
        for _ in range(rng.randint(0, 5)):
            kept = sorted(rng.sample(range(n_kept[r]), rng.randint(1, n_kept[r])))
            row, crow = [-2] * n, [0] * n
            for i, k in enumerate(kept):
                row[i] = rng.choice([-1, 0, 0, 1, 2, 3, 5])
                crow[i] = k
            cells.append(row)
            cand.append(crow)
            rec.append(r)
    cells, rec, cand = np.array(cells, np.int32), np.array(rec, np.int32), np.array(cand, np.int8)
    emeta, esums = W.vote_groups(cells, rec, weight, cand)
    for dtype in (torch.int8, torch.int32):
        meta, sums = K.weighted_vote_groups(torch.from_numpy(cells).to(dtype).cuda(), torch.from_numpy(rec).cuda(),
                                            torch.from_numpy(weight).cuda(), torch.from_numpy(cand).cuda())
        assert np.array_equal(meta.cpu().numpy().view(np.uint32), emeta), (n, dtype)
        assert np.array_equal(sums.cpu().numpy().view(np.uint32), esums.view(np.uint32)), (n, dtype)
    # without a cand map cell c is candidate c
    full = np.array([[rng.choice([-1, 0, 1, 2]) if i < n_kept[r] else -2 for i in range(n)] for r in rec], dtype=np.int32)
    emeta, esums = W.vote_groups(full, rec, weight)
    meta, sums = K.weighted_vote_groups(torch.from_numpy(full).cuda(), torch.from_numpy(rec).cuda(), torch.from_numpy(weight).cuda())
    assert np.array_equal(meta.cpu().numpy().view(np.uint32), emeta)
    assert np.array_equal(sums.cpu().numpy().view(np.uint32), esums.view(np.uint32))


def _mixed_records():
    """Device-path records (flat, nested, S32) and records the device path declines (lists, differing keys, phrases)."""
    from oracle.gen_golden import random_list_records
    from tests.test_weighted_host_logic import _records
    out = [recs for recs in _records().values()]
    lists = [[json.dumps(v) for v in rec] for rec in random_list_records(31, 150)]
    rng = random.Random(4)
    differing = []
    for _ in range(60):
        n = rng.choice([2, 3, 5])
        differing.append([json.dumps({k: rng.choice(["a", "b", "B!"]) for k in rng.sample(["x", "y", "z"], rng.randint(1, 3))})
                          for _ in range(n)])
    return [r for recs in out for r in recs] + lists + differing


def _expected(texts, lp):
    """The weighted oracle after the list alignment pre-pass the product runs (pinned on the reference's goldens)."""
    import logging

    from k_llms_b200.utils.consensus_utils import recursive_list_alignments
    from k_llms_b200.utils.consolidation import _safe_parse_content
    contents = [_safe_parse_content(t) for t in texts if t]
    aligned = None
    if len(contents) >= 2:
        logging.disable(logging.CRITICAL)
        try:
            aligned, _ = recursive_list_alignments(contents, "embeddings", raising_embeddings, None, 0.51)
        finally:
            logging.disable(logging.NOTSET)
    return W.expected(texts, lp, embed=raising_embeddings, aligned=aligned)


def test_consolidate_contents_batch_weighted(torch):
    from k_llms_b200.utils.consensus_utils import ConsensusSettings
    from k_llms_b200.utils.consolidation import consolidate_contents_batch
    lk = ConsensusSettings(candidate_weighting="likelihood")
    recs = _mixed_records()
    rng = random.Random(8)
    lps = [W.random_logprobs(rng, len(t), scale=rng.choice([0.1, 1.0, 40.0])) for t in recs]
    got = consolidate_contents_batch(recs, lk, raising_embeddings, logprobs=lps)
    for texts, lp, (content, lik) in zip(recs, lps, got):
        ec, el = _expected(texts, lp)
        assert (content, json.dumps(lik)) == (ec, el), (texts, lp)
    # equal sequence sums: byte-identical to the uniform consolidation
    eq = consolidate_contents_batch(recs, lk, raising_embeddings, logprobs=[W.equal_logprobs(len(t)) for t in recs])
    assert eq == consolidate_contents_batch(recs, ConsensusSettings(), raising_embeddings)


def _config4_batch(R, n, seed):
    """R records of n candidate texts (4 vote fields and one number, 8 spellings per field; every text padded to one length,
    so the blob is built by indexing) and 8..64 token logprobs per candidate."""
    from k_llms_b200 import _native as K
    rng = np.random.default_rng(seed)
    pool = []
    for i in range(64):
        d = {"city": ["Paris", "paris", "Lyon", "Nice"][i % 4], "ok": bool(i & 4), "tier": ["gold", "Silver"][(i >> 3) & 1],
             "code": ["a1", "b2", "A1"][i % 3], "n": i % 5}
        pool.append(json.dumps(d))
    L = max(len(t) for t in pool)
    pool_bytes = np.frombuffer("".join(t.ljust(L) for t in pool).encode(), dtype=np.uint8).reshape(64, L)
    pick = rng.integers(0, 64, R * n)
    blob = K.pinned_empty((R * n * L,), np.uint8)
    blob[:] = pool_bytes[pick].reshape(-1)
    off = np.arange(R * n + 1, dtype=np.int64) * L
    lens = rng.integers(8, 65, R * n)
    lp_off = np.zeros(R * n + 1, dtype=np.int64)
    np.cumsum(lens, out=lp_off[1:])
    lp = K.pinned_empty((int(lp_off[-1]),), np.float32)
    lp[:] = -rng.exponential(0.5, int(lp_off[-1])).astype(np.float32)
    texts = [t.ljust(L) for t in pool]
    return blob, off, lp, lp_off, pick, texts


def test_config4_shaped_weighted_entry(torch):
    from k_llms_b200 import _native as K
    R, n = 256 * 1024, 32
    blob, off, lp, lp_off, pick, pool = _config4_batch(R, n, 20261017)
    uni = K.consolidate_json_packed(blob, off, n)
    # equal logprobs: every weight is 1.0f, the output is the uniform one byte for byte
    eq_off = np.arange(R * n + 1, dtype=np.int64) * 8  # 8 equal tokens per candidate: equal sums
    eqw = K.consolidate_json_packed(blob, off, n, logprobs=(np.full(R * n * 8, -0.5, np.float32), eq_off))
    assert (uni.status == 0).all() and (eqw.status == 0).all()
    assert uni.pairs() == eqw.pairs()
    assert eqw.stats.input_bytes == int(off[-1]) + R * n * 8 * 4
    eqw.close()
    # random logprobs: a seeded sample against the oracle
    res = K.consolidate_json_packed(blob, off, n, logprobs=(lp, lp_off))
    assert (res.status == 0).all()
    rng = random.Random(3)
    for r in rng.sample(range(R), 300):
        texts = [pool[int(k)] for k in pick[r * n:(r + 1) * n]]
        lps = [lp[lp_off[r * n + c]:lp_off[r * n + c + 1]].tolist() for c in range(n)]
        ec, el = W.expected(texts, lps, embed=raising_embeddings)
        assert (res.content(r), res.likelihoods(r)) == (ec, el), r
    changed = sum(res.content(r) != uni.content(r) for r in range(0, R, 97))
    assert changed > 0  # the weights decide some records differently
    res.close()
    uni.close()


def test_client_create_with_likelihood_weighting(torch):
    from k_llms_b200.client import KLLMs
    from k_llms_b200.utils.consensus_utils import ConsensusSettings
    from tests.test_weighted_host_logic import StubOpenAI, _completion
    contents = [json.dumps({"city": "Paris", "ok": True})] * 2 + [json.dumps({"city": "Lyon", "ok": False})] * 3
    lps = [[-0.01, -0.02]] * 2 + [[-3.0, -2.5]] * 3
    stub = StubOpenAI(_completion(contents, lps))
    k = KLLMs(api_key="test")
    k._client = stub
    out = k.chat.completions.create(messages=[{"role": "user", "content": "?"}], model="m", n=5,
                                    consensus_settings=ConsensusSettings(candidate_weighting="likelihood"))
    assert stub.requests[-1]["logprobs"] is True
    ec, el = W.expected(contents, lps)
    assert out.choices[0].message.content == ec == json.dumps({"city": "Paris", "ok": True})
    assert json.dumps(out.likelihoods) == el
    uniform = k.chat.completions.create(messages=[{"role": "user", "content": "?"}], model="m", n=5)
    assert json.loads(uniform.choices[0].message.content) == {"city": "Lyon", "ok": False}
