"""ctypes binding of libkllms_b200.so — the C ABI declared in include/kllms_b200.h.

This is the ONLY compute path of the package: there is no CPU fallback.  If the shared library has not
been built (`python -c "import __graft_entry__ as g; g.build()"` or `make -C k_llms_b200/csrc`) or no
sm_100 device is visible, the functions below raise — loudly — instead of computing on the host.

torch is used for device memory and streams only (plumbing); the ABI itself takes raw pointers.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KLLMS_B200_LIB") or os.path.join(_HERE, "libkllms_b200.so")

KC_OK, KC_EINVAL, KC_ECUDA, KC_ENODEV, KC_ENOMEM = 0, -1, -2, -3, -4
MAX_CANDIDATES = 64
CODE_NONE, CODE_ABSENT = -1, -2
F64_NONE_BITS = 0x7FF8C0DE00000000
F64_ABSENT_BITS = 0x7FF8C0DF00000000
FLAG_HAS_VALUE, FLAG_SINGLE, FLAG_TIE, FLAG_NO_FINITE = 1, 2, 4, 8
OUT_LOCAL, OUT_MULTIMEM, OUT_PEERS = 0, 1, 2

EXPORTS = (
    "kc_version", "kc_last_error", "kc_device_count", "kc_sm_count", "kc_set_device", "kc_vote_i32", "kc_numeric_f64", "kc_vote_i32_ex", "kc_numeric_f64_ex", "kc_vote_i8", "kc_consensus_host_i8", "kc_consolidate_json", "kc_free_strings", "kc_levenshtein", "kc_medoid_str", "kc_medoid_str_host", "kc_align_json", "kc_debug_similarity_json", "kc_debug_lsap", "kc_json_plan", "kc_json_inputs", "kc_json_emit", "kc_json_free", "kc_vote_i32_peers", "kc_numeric_f64_peers", "kc_vote_i32_peers_packed",
    "kc_confidence_f64", "kc_logprob_sum_f32", "kc_weighted_vote_i32", "kc_consensus_host", "kc_host_alloc", "kc_host_free",
    "kc_consolidate_json_packed", "kc_json_result_view", "kc_json_result_free", "kc_debug_jsongpu_plan", "kc_debug_jsongpu_inputs",
    "kc_debug_jsongpu_emit", "kc_debug_jsongpu_medoid_inputs", "kc_debug_jsongpu_set_medoid", "kc_debug_jsongpu_free", "kc_debug_parse_doubles", "kc_debug_float_reprs", "kc_debug_round5", "kc_debug_s32_texts", "kc_push_results", "kc_vote_i32_wire", "kc_medoid_str_method",
    "kc_candidate_weights_f32", "kc_weighted_vote_groups_i8", "kc_weighted_vote_groups_i32", "kc_consolidate_json_packed_weighted",
    "kc_debug_jsongpu_vote_records", "kc_debug_jsongpu_emit_weighted",
)


class NativeError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"libkllms_b200: {what} (code {code})")
        self.code = code


_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """dlopen the library and declare prototypes.  Raises if it is missing: no silent fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the sm_100a library first (make -C k_llms_b200/csrc, or "
            "__graft_entry__.build()).  k_llms_b200 has no CPU fallback for the consensus hot path.")
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i32, i64, f64 = c.c_void_p, c.c_int32, c.c_int64, c.c_double
    lib.kc_version.restype = c.c_int
    lib.kc_last_error.restype = c.c_char_p
    lib.kc_device_count.restype = c.c_int
    lib.kc_sm_count.argtypes = [c.c_int]
    lib.kc_set_device.argtypes = [c.c_int]
    lib.kc_vote_i32.argtypes = [vp, i64, i32, vp, i32, vp, vp, vp]
    lib.kc_numeric_f64.argtypes = [vp, i64, i32, f64, f64, vp, vp, vp]
    lib.kc_vote_i32_ex.argtypes = [vp, i64, i32, vp, i32, vp, vp, c.c_uint32, vp]
    lib.kc_numeric_f64_ex.argtypes = [vp, i64, i32, f64, f64, vp, vp, c.c_uint32, vp]
    lib.kc_confidence_f64.argtypes = [vp, i64, i32, vp, vp, vp]
    lib.kc_logprob_sum_f32.argtypes = [vp, vp, i64, vp, vp]
    lib.kc_weighted_vote_i32.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, vp, vp]
    lib.kc_candidate_weights_f32.argtypes = [vp, i64, i32, vp, vp]
    lib.kc_weighted_vote_groups_i8.argtypes = [vp, i64, i32, vp, vp, vp, vp, vp, vp]
    lib.kc_weighted_vote_groups_i32.argtypes = lib.kc_weighted_vote_groups_i8.argtypes
    lib.kc_consolidate_json_packed_weighted.argtypes = [vp, vp, vp, vp, i64, i32, f64, f64, c.c_int, i32, c.c_uint32, c.POINTER(vp)]
    lib.kc_debug_jsongpu_vote_records.argtypes = [vp, c.POINTER(vp)]
    lib.kc_debug_jsongpu_emit_weighted.argtypes = [vp, vp, vp, vp, vp] + [c.POINTER(vp)] * 4
    lib.kc_consensus_host.argtypes = [vp, i32, vp, vp, i32, i64, i32, f64, f64, vp, vp, vp, vp, c.c_int, vp]
    lib.kc_consensus_host_i8.argtypes = lib.kc_consensus_host.argtypes
    lib.kc_vote_i8.argtypes = [vp, i64, i32, vp, i32, vp, vp, vp]
    lib.kc_consolidate_json.argtypes = [vp, vp, i64, i32, f64, f64, c.c_int, i32, vp, vp, vp]
    lib.kc_consolidate_json.restype = c.c_int
    lib.kc_vote_i32_peers.argtypes = [vp, i64, i32, vp, i32, vp, vp, i32, vp, vp]
    lib.kc_numeric_f64_peers.argtypes = [vp, i64, i32, f64, f64, vp, vp, i32, vp, vp]
    lib.kc_vote_i32_peers_packed.argtypes = [vp, i64, i32, vp, i32, vp, vp, vp, i32, vp, vp, vp]
    lib.kc_vote_i32_peers.restype = lib.kc_numeric_f64_peers.restype = lib.kc_vote_i32_peers_packed.restype = c.c_int
    lib.kc_json_plan.argtypes = [vp, vp, i64, i32, i32, c.POINTER(vp)]
    lib.kc_json_inputs.argtypes = [vp] + [vp] * 9
    lib.kc_json_emit.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.kc_json_plan.restype = lib.kc_json_inputs.restype = lib.kc_json_emit.restype = c.c_int
    lib.kc_json_free.argtypes = [vp]
    lib.kc_json_free.restype = None
    lib.kc_align_json.argtypes = [c.POINTER(c.c_char_p), vp, i32, f64, c.POINTER(c.c_char_p)]
    lib.kc_align_json.restype = c.c_int
    lib.kc_debug_similarity_json.argtypes = [c.c_char_p, c.c_char_p, c.POINTER(c.c_double)]
    lib.kc_debug_lsap.argtypes = [i32, i32, vp, vp, vp]
    lib.kc_debug_similarity_json.restype = lib.kc_debug_lsap.restype = c.c_int
    lib.kc_medoid_str_host.argtypes = [vp, i64, vp, vp, i64, i32, vp, vp, c.c_int]
    lib.kc_medoid_str_host.restype = c.c_int
    lib.kc_medoid_str.argtypes = [vp, vp, vp, i64, i32, vp, vp, vp]
    lib.kc_medoid_str.restype = c.c_int
    lib.kc_medoid_str_method.argtypes = [vp, vp, vp, i64, i32, i32, vp, vp, vp]
    lib.kc_medoid_str_method.restype = c.c_int
    lib.kc_levenshtein.argtypes = [c.c_char_p, i32, c.c_char_p, i32]
    lib.kc_levenshtein.restype = i32
    lib.kc_free_strings.argtypes = [vp, i64]
    lib.kc_free_strings.restype = None
    lib.kc_consolidate_json_packed.argtypes = [vp, vp, i64, i32, f64, f64, c.c_int, i32, c.c_uint32, c.POINTER(vp)]
    lib.kc_json_result_view.argtypes = [vp] + [c.POINTER(vp)] * 7 + [vp]
    lib.kc_json_result_free.argtypes = [vp]
    lib.kc_json_result_free.restype = None
    lib.kc_debug_jsongpu_plan.argtypes = [vp, vp, i64, i32, c.POINTER(vp)]
    lib.kc_debug_jsongpu_inputs.argtypes = [vp] + [vp] * 5
    lib.kc_debug_jsongpu_emit.argtypes = [vp, vp, vp, vp] + [c.POINTER(vp)] * 4
    lib.kc_debug_jsongpu_medoid_inputs.argtypes = [vp] + [c.POINTER(vp)] * 3 + [c.POINTER(i64)]
    lib.kc_debug_jsongpu_set_medoid.argtypes = [vp, vp, vp]
    lib.kc_debug_jsongpu_medoid_inputs.restype = lib.kc_debug_jsongpu_set_medoid.restype = c.c_int
    lib.kc_debug_jsongpu_free.argtypes = [vp]
    lib.kc_debug_jsongpu_free.restype = None
    lib.kc_debug_parse_doubles.argtypes = [vp, vp, i64, vp, vp]
    lib.kc_debug_float_reprs.argtypes = [vp, i64, vp, vp]
    lib.kc_debug_round5.argtypes = [vp, i64, vp]
    lib.kc_debug_s32_texts.argtypes = [c.c_uint64, i64, i32, i32, vp, i64, vp]
    lib.kc_debug_s32_texts.restype = c.c_int
    lib.kc_push_results.argtypes = [vp, vp, i64, vp, vp, i64, vp, vp, vp, i32, i32, vp, vp, i32, vp]
    lib.kc_push_results.restype = c.c_int
    lib.kc_vote_i32_wire.argtypes = [vp, i64, i32, vp, i32, vp, vp, vp, i32, i32, vp, vp, vp]
    lib.kc_vote_i32_wire.restype = c.c_int
    for name in ("kc_consolidate_json_packed", "kc_consolidate_json_packed_weighted", "kc_debug_jsongpu_vote_records",
                 "kc_debug_jsongpu_emit_weighted", "kc_candidate_weights_f32", "kc_weighted_vote_groups_i8", "kc_weighted_vote_groups_i32",
                 "kc_json_result_view", "kc_debug_jsongpu_plan", "kc_debug_jsongpu_inputs",
                 "kc_debug_jsongpu_emit", "kc_debug_parse_doubles", "kc_debug_float_reprs", "kc_debug_round5"):
        getattr(lib, name).restype = c.c_int
    lib.kc_host_alloc.argtypes = [c.c_uint64]
    lib.kc_host_alloc.restype = vp
    lib.kc_host_free.argtypes = [vp]
    lib.kc_host_free.restype = None
    for name in ("kc_sm_count", "kc_set_device", "kc_vote_i32", "kc_numeric_f64", "kc_confidence_f64", "kc_logprob_sum_f32",
                 "kc_weighted_vote_i32", "kc_vote_i32_ex", "kc_numeric_f64_ex", "kc_vote_i8", "kc_consensus_host_i8", "kc_vote_i8", "kc_consensus_host_i8", "kc_consolidate_json", "kc_free_strings", "kc_levenshtein", "kc_medoid_str", "kc_medoid_str_host", "kc_align_json", "kc_debug_similarity_json", "kc_debug_lsap", "kc_json_plan", "kc_json_inputs", "kc_json_emit", "kc_json_free", "kc_vote_i32_peers", "kc_numeric_f64_peers", "kc_vote_i32_peers_packed",
                 "kc_consensus_host"):
        getattr(lib, name).restype = c.c_int
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != KC_OK:
        raise NativeError(rc, load().kc_last_error().decode(errors="replace"))


def _require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("k_llms_b200 needs a CUDA (sm_100a) device: the consensus hot path has no CPU fallback")
    return torch


def _stream_ptr(torch, stream) -> int:
    s = stream if stream is not None else torch.cuda.current_stream()
    return int(s.cuda_stream)


def _bind(torch, t) -> None:
    check(load().kc_set_device(t.device.index if t.device.index is not None else torch.cuda.current_device()))


def vote(codes, none_code=None, stream=None) -> Tuple["torch.Tensor", "torch.Tensor"]:
    """K1 on device tensors.  codes: int32 [G, n] (cuda, contiguous); none_code: int32 [F] or None.
    Returns (win_code int32 [G], meta int32 [G] holding the packed uint32 word)."""
    torch = _require_cuda()
    assert codes.is_cuda and codes.dtype == torch.int32 and codes.dim() == 2 and codes.is_contiguous()
    G, n = codes.shape
    win = torch.empty(G, dtype=torch.int32, device=codes.device)
    meta = torch.empty(G, dtype=torch.int32, device=codes.device)
    nf = 0
    nc_ptr = None
    if none_code is not None:
        assert none_code.is_cuda and none_code.dtype == torch.int32 and none_code.is_contiguous()
        nf = none_code.numel()
        assert G % nf == 0, "n_groups must be a whole number of records"
        nc_ptr = none_code.data_ptr()
    _bind(torch, codes)
    check(load().kc_vote_i32(codes.data_ptr(), G, n, nc_ptr, nf, win.data_ptr(), meta.data_ptr(), _stream_ptr(torch, stream)))
    return win, meta


def vote_i8(codes, none_code=None, stream=None):
    """K1 on compact int8 cells (cuda int8 [G, n])."""
    torch = _require_cuda()
    assert codes.is_cuda and codes.dtype == torch.int8 and codes.dim() == 2 and codes.is_contiguous()
    G, n = codes.shape
    win = torch.empty(G, dtype=torch.int32, device=codes.device)
    meta = torch.empty(G, dtype=torch.int32, device=codes.device)
    nf, nc_ptr = 0, None
    if none_code is not None:
        nf, nc_ptr = none_code.numel(), none_code.data_ptr()
    _bind(torch, codes)
    check(load().kc_vote_i8(codes.data_ptr(), G, n, nc_ptr, nf, win.data_ptr(), meta.data_ptr(), _stream_ptr(torch, stream)))
    return win, meta


def numeric(vals, rel_eps: float = 0.03, abs_eps: float = 1e-6, stream=None):
    """K2 on device tensors.  vals: float64 [G, n].  Returns (value float64 [G], meta int32 [G])."""
    torch = _require_cuda()
    assert vals.is_cuda and vals.dtype == torch.float64 and vals.dim() == 2 and vals.is_contiguous()
    G, n = vals.shape
    value = torch.empty(G, dtype=torch.float64, device=vals.device)
    meta = torch.empty(G, dtype=torch.int32, device=vals.device)
    _bind(torch, vals)
    check(load().kc_numeric_f64(vals.data_ptr(), G, n, float(rel_eps), float(abs_eps), value.data_ptr(), meta.data_ptr(),
                                _stream_ptr(torch, stream)))
    return value, meta


def confidence(meta, numeric_kind: bool, pvf=None, stream=None):
    """Python-round(x,5)-exact confidences from result words.  meta int32 [G]; pvf float64 [G] or None."""
    torch = _require_cuda()
    assert meta.is_cuda and meta.dtype == torch.int32 and meta.is_contiguous()
    conf = torch.empty(meta.numel(), dtype=torch.float64, device=meta.device)
    pv = None
    if pvf is not None:
        assert pvf.is_cuda and pvf.dtype == torch.float64 and pvf.numel() == meta.numel() and pvf.is_contiguous()
        pv = pvf.data_ptr()
    _bind(torch, meta)
    check(load().kc_confidence_f64(meta.data_ptr(), meta.numel(), 1 if numeric_kind else 0, pv, conf.data_ptr(),
                                   _stream_ptr(torch, stream)))
    return conf


def logprob_sum(logprobs, offsets, stream=None):
    """K3: fp32 per-sequence sums.  logprobs float32 [T], offsets int64 [S+1] -> float32 [S]."""
    torch = _require_cuda()
    assert logprobs.is_cuda and logprobs.dtype == torch.float32 and offsets.dtype == torch.int64 and offsets.is_cuda
    out = torch.empty(offsets.numel() - 1, dtype=torch.float32, device=logprobs.device)
    _bind(torch, logprobs)
    check(load().kc_logprob_sum_f32(logprobs.data_ptr(), offsets.data_ptr(), out.numel(), out.data_ptr(),
                                    _stream_ptr(torch, stream)))
    return out


def weighted_vote(codes, seq_logprob, none_code=None, stream=None):
    """K3b: likelihood-weighted vote.  codes int32 [R, F, n], seq_logprob float32 [R, n] (cuda).
    Returns (win_code int32 [R*F], meta int32 [R*F], weight float32 [R*F])."""
    torch = _require_cuda()
    assert codes.is_cuda and codes.dtype == torch.int32 and codes.dim() == 3 and codes.is_contiguous()
    R, F, n = codes.shape
    assert seq_logprob.is_cuda and seq_logprob.dtype == torch.float32 and tuple(seq_logprob.shape) == (R, n)
    assert seq_logprob.is_contiguous()
    win = torch.empty(R * F, dtype=torch.int32, device=codes.device)
    meta = torch.empty(R * F, dtype=torch.int32, device=codes.device)
    weight = torch.empty(R * F, dtype=torch.float32, device=codes.device)
    nc = None
    if none_code is not None:
        assert none_code.is_cuda and none_code.dtype == torch.int32 and none_code.numel() == F
        nc = none_code.data_ptr()
    _bind(torch, codes)
    check(load().kc_weighted_vote_i32(codes.data_ptr(), seq_logprob.data_ptr(), R, F, n, nc, win.data_ptr(), meta.data_ptr(),
                                      weight.data_ptr(), _stream_ptr(torch, stream)))
    return win, meta, weight


def candidate_weights(seq_logprob, stream=None):
    """Candidate weights of likelihood-weighted consolidation (self-defined, DESIGN.md §5): seq_logprob float32 [R, n] (cuda) ->
    float32 [R, n], w_c = kexp(s_c - max_k s_k) per record (K3b's weight pre-pass)."""
    torch = _require_cuda()
    assert seq_logprob.is_cuda and seq_logprob.dtype == torch.float32 and seq_logprob.dim() == 2 and seq_logprob.is_contiguous()
    R, n = seq_logprob.shape
    out = torch.empty(R, n, dtype=torch.float32, device=seq_logprob.device)
    _bind(torch, seq_logprob)
    check(load().kc_candidate_weights_f32(seq_logprob.data_ptr(), R, n, out.data_ptr(), _stream_ptr(torch, stream)))
    return out


def weighted_vote_groups(cells, group_record, weight, cand=None, stream=None):
    """Likelihood-weighted vote over irregular groups (self-defined, DESIGN.md §5).  cells int8 or int32 [G, n] (K1's coding),
    group_record int32 [G], weight float32 [R, n] (candidate_weights), cand int8 [G, n] or None (cell c is candidate c); all cuda.
    Returns (meta int32 [G] holding K1's packed uint32 word, sums float32 [G, 2] = (W_win, W_present))."""
    torch = _require_cuda()
    assert cells.is_cuda and cells.dtype in (torch.int8, torch.int32) and cells.dim() == 2 and cells.is_contiguous()
    G, n = cells.shape
    assert group_record.is_cuda and group_record.dtype == torch.int32 and group_record.numel() == G and group_record.is_contiguous()
    assert weight.is_cuda and weight.dtype == torch.float32 and weight.dim() == 2 and weight.shape[1] == n and weight.is_contiguous()
    cp = None
    if cand is not None:
        assert cand.is_cuda and cand.dtype == torch.int8 and tuple(cand.shape) == (G, n) and cand.is_contiguous()
        cp = cand.data_ptr()
    meta = torch.empty(G, dtype=torch.int32, device=cells.device)
    sums = torch.empty(G, 2, dtype=torch.float32, device=cells.device)
    entry = load().kc_weighted_vote_groups_i8 if cells.dtype == torch.int8 else load().kc_weighted_vote_groups_i32
    _bind(torch, cells)
    check(entry(cells.data_ptr(), G, n, group_record.data_ptr(), cp, weight.data_ptr(), meta.data_ptr(), sums.data_ptr(),
                _stream_ptr(torch, stream)))
    return meta, sums


def consensus_host(codes, none_code, vals, rel_eps=0.03, abs_eps=1e-6, device=0, out=None):
    """End-to-end entry with HOST numpy arrays (ideally backed by pinned memory).
    codes int32 [N, Fv, n] or None; none_code int32 [Fv] or None; vals float64 [N, Fx, n] or None.
    Returns dict(win_code, vote_meta, value, num_meta) of numpy arrays."""
    import numpy as np
    lib = load()
    N = n = Fv = Fx = 0
    if codes is not None:
        assert codes.dtype in (np.int32, np.int8) and codes.ndim == 3 and codes.flags.c_contiguous
        N, Fv, n = codes.shape
    if vals is not None:
        assert vals.dtype == np.float64 and vals.ndim == 3 and vals.flags.c_contiguous
        N2, Fx, n2 = vals.shape
        assert codes is None or (N2 == N and n2 == n)
        N, n = N2, n2
    out = out or {}
    win = out.get("win_code") if "win_code" in out else np.empty((N, Fv), dtype=np.int32)
    vmeta = out.get("vote_meta") if "vote_meta" in out else np.empty((N, Fv), dtype=np.uint32)
    value = out.get("value") if "value" in out else np.empty((N, Fx), dtype=np.float64)
    nmeta = out.get("num_meta") if "num_meta" in out else np.empty((N, Fx), dtype=np.uint32)
    if none_code is not None:
        none_code = np.ascontiguousarray(none_code, dtype=np.int32)
        assert none_code.size == Fv
    p = lambda a: a.ctypes.data if a is not None and a.size else None  # noqa: E731
    ms = ctypes.c_float(0.0)
    entry = lib.kc_consensus_host_i8 if (codes is not None and codes.dtype == np.int8) else lib.kc_consensus_host
    check(entry(p(codes), Fv, p(none_code), p(vals), Fx, N, n, float(rel_eps), float(abs_eps), p(win), p(vmeta),
                p(value), p(nmeta), device, ctypes.addressof(ms)))
    return {"win_code": win, "vote_meta": vmeta, "value": value, "num_meta": nmeta, "device_ms": float(ms.value)}


SIM_METHODS = {"levenshtein": 0, "embeddings": 0, "jaccard": 1, "hamming": 2}  # "embeddings": pairs the planner sends here are Levenshtein pairs


def medoid_str(chars, str_off, grp_off, max_group=MAX_CANDIDATES, stream=None, method: str = "levenshtein"):
    """K4 on device tensors: chars uint8 [C], str_off int32 [S+1], grp_off int32 [G+1], max_group = largest group ->
    (best index int32 [G], mean similarity float64 [G]); method = the reference's string_similarity_method."""
    torch = _require_cuda()
    assert chars.is_cuda and chars.dtype == torch.uint8 and str_off.dtype == torch.int32 and grp_off.dtype == torch.int32
    G = grp_off.numel() - 1
    idx = torch.empty(G, dtype=torch.int32, device=chars.device)
    avg = torch.empty(G, dtype=torch.float64, device=chars.device)
    _bind(torch, chars)
    check(load().kc_medoid_str_method(chars.data_ptr(), str_off.data_ptr(), grp_off.data_ptr(), G, max(2, int(max_group)),
                                      SIM_METHODS[method], idx.data_ptr(), avg.data_ptr(), _stream_ptr(torch, stream)))
    return idx, avg


def align_json(values, min_support_ratio: float):
    """H2: the alignment pre-pass (recursive_list_alignments, default similarity method) of ONE record in native code.
    values: n JSON-serialisable candidate values.  Returns the aligned values, or None when the record needs the Python
    pre-pass (long string pairs that go to the embeddings service, non-ASCII text, values json cannot carry)."""
    import json
    n = len(values)
    if n == 0:
        return None
    # Precondition: the values look like json.loads output as far as OBJECT IDENTITY goes.  The reference's majority ordering
    # finds an aligned cell's source position by id() (majority_sorting.py:14-17), and the native code restates CPython's
    # behaviour for freshly parsed values (True / False / ints in [-5, 256] / one-character strings are shared objects,
    # everything else is distinct).  A list holding the SAME longer string / float / big int object twice (built in Python, or
    # deep-copied) breaks that: leave such records to the Python pre-pass, which sees the real identities.
    def shared_identity(v) -> bool:
        if isinstance(v, dict):
            return any(shared_identity(x) for x in v.values())
        if isinstance(v, list):
            seen = set()
            for x in v:
                if (isinstance(x, str) and len(x) > 1) or isinstance(x, float) or (isinstance(x, int) and not isinstance(x, bool) and not -5 <= x <= 256):
                    if id(x) in seen:
                        return True
                    seen.add(id(x))
            return any(shared_identity(x) for x in v)
        return False
    if any(shared_identity(v) for v in values):
        return None
    try:
        texts = (ctypes.c_char_p * n)(*[json.dumps(v).encode("ascii") for v in values])
    except (TypeError, ValueError):
        return None
    out = (ctypes.c_char_p * n)()
    rc = load().kc_align_json(texts, None, n, float(min_support_ratio), out)
    if rc != 0:
        return None
    try:
        return [json.loads(out[i]) for i in range(n)]
    finally:
        load().kc_free_strings(out, n)


def levenshtein(a: str, b: str) -> int:
    """Edit distance through the native library (code points must be Latin-1; callers pass normalised ASCII)."""
    ba, bb = a.encode("latin-1"), b.encode("latin-1")
    return int(load().kc_levenshtein(ba, len(ba), bb, len(bb)))


def consolidate_json(records, rel_eps: float = 0.03, abs_eps: float = 1e-6, device: int = 0, threads: int = 0):
    """H1: native consolidation of records of scalars, nested objects and lists (default settings).  records: list of lists of n candidate content strings.
    Returns a list of (content_str, likelihoods_json_str) or None where the record needs the Python path."""
    lib = load()
    R = len(records)
    if R == 0:
        return []
    n = len(records[0])
    assert all(len(r) == n for r in records), "every record needs the same number of candidates"
    blobs = [t.encode("utf-8") for r in records for t in r]
    texts = (ctypes.c_char_p * (R * n))(*blobs)
    lens = (ctypes.c_int64 * (R * n))(*[len(b) for b in blobs])
    out_c = (ctypes.c_void_p * R)()
    out_l = (ctypes.c_void_p * R)()
    status = (ctypes.c_uint8 * R)()
    check(lib.kc_consolidate_json(ctypes.cast(texts, ctypes.c_void_p), ctypes.cast(lens, ctypes.c_void_p), R, n, float(rel_eps),
                                  float(abs_eps), device, threads, ctypes.cast(out_c, ctypes.c_void_p),
                                  ctypes.cast(out_l, ctypes.c_void_p), ctypes.cast(status, ctypes.c_void_p)))
    res = []
    for i in range(R):
        if status[i] == 0:
            res.append((ctypes.string_at(out_c[i]).decode("ascii"), ctypes.string_at(out_l[i]).decode("ascii")))
        else:
            res.append(None)
    lib.kc_free_strings(ctypes.cast(out_c, ctypes.c_void_p), R)
    lib.kc_free_strings(ctypes.cast(out_l, ctypes.c_void_p), R)
    return res


def pinned_empty(shape, dtype):
    """numpy array backed by page-locked memory from kc_host_alloc (freed when the array is collected)."""
    import numpy as np
    lib = load()
    dt = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dt.itemsize
    ptr = lib.kc_host_alloc(max(nbytes, 1))
    if not ptr:
        raise MemoryError(f"kc_host_alloc({nbytes}) failed")
    buf = (ctypes.c_uint8 * max(nbytes, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
    import weakref
    weakref.finalize(buf, lib.kc_host_free, ptr)
    return arr


class JsonStats(ctypes.Structure):
    """kc_json_stats (include/kllms_b200.h)."""
    _fields_ = [(k, ctypes.c_int64) for k in ("n_records", "n_device", "n_host", "n_python", "input_bytes", "output_bytes")] + \
               [("chunks", ctypes.c_int32), ("streams", ctypes.c_int32)] + \
               [(k, ctypes.c_double) for k in ("h2d_ms", "plan_ms", "kernel_ms", "emit_ms", "d2h_ms", "device_path_wall_ms",
                                               "host_path_wall_ms", "wall_ms")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


JSON_DEVICE_ONLY = 1


def pack_texts(records, pinned: bool = True):
    """records: list of lists of n candidate content strings -> (blob uint8 array, off int64 array [R*n+1], n): the packed
    form kc_consolidate_json_packed takes (blob in page-locked memory when `pinned`)."""
    import numpy as np
    R = len(records)
    n = len(records[0]) if R else 0
    assert all(len(r) == n for r in records), "every record needs the same number of candidates"
    enc = [t.encode("utf-8") for r in records for t in r]
    off = np.zeros(R * n + 1, dtype=np.int64)
    if enc:
        np.cumsum(np.fromiter((len(b) for b in enc), dtype=np.int64, count=len(enc)), out=off[1:])
    total = int(off[-1])
    blob = pinned_empty((max(total, 1),), np.uint8) if pinned else np.empty(max(total, 1), dtype=np.uint8)
    if total:
        blob[:total] = np.frombuffer(b"".join(enc), dtype=np.uint8)
    return blob, off, n


class PackedResult:
    """View of a kc_json_result: `content(r)` / `likelihoods(r)` are the texts of record r (None when status is 1)."""

    def __init__(self, handle, R):
        import numpy as np
        self._h, self.R = handle, R
        lib = load()
        ptrs = [ctypes.c_void_p() for _ in range(7)]
        self.stats = JsonStats()
        check(lib.kc_json_result_view(handle, *[ctypes.byref(p) for p in ptrs], ctypes.addressof(self.stats)))
        as_i64 = lambda p: np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_int64)), shape=(R,)) if R else np.zeros(0, np.int64)  # noqa: E731
        as_u8 = lambda p: np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(R,)) if R else np.zeros(0, np.uint8)  # noqa: E731
        self._text = ptrs[0].value or 0
        self.c_off, self.c_len, self.l_off, self.l_len = as_i64(ptrs[1]), as_i64(ptrs[2]), as_i64(ptrs[3]), as_i64(ptrs[4])
        self.status, self.why = as_u8(ptrs[5]), as_u8(ptrs[6])

    def content(self, r):
        return None if self.status[r] == 1 else ctypes.string_at(self._text + int(self.c_off[r]), int(self.c_len[r])).decode("ascii")

    def likelihoods(self, r):
        return None if self.status[r] == 1 else ctypes.string_at(self._text + int(self.l_off[r]), int(self.l_len[r])).decode("ascii")

    def pairs(self):
        return [None if self.status[r] == 1 else (self.content(r), self.likelihoods(r)) for r in range(self.R)]

    def close(self):
        if self._h is not None:
            load().kc_json_result_free(self._h)
            self._h = None

    def __del__(self):
        self.close()


def pack_logprobs(records_logprobs, pinned: bool = True):
    """records_logprobs: per record, per candidate a sequence of token logprobs (record-major, like pack_texts' records) ->
    (lp float32 array, lp_off int64 [R*n+1]): the packed form kc_consolidate_json_packed_weighted takes (lp in page-locked
    memory when `pinned`)."""
    import numpy as np
    seqs = [s for rec in records_logprobs for s in rec]
    lp_off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if seqs:
        np.cumsum(np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs)), out=lp_off[1:])
    total = int(lp_off[-1])
    lp = pinned_empty((max(total, 1),), np.float32) if pinned else np.empty(max(total, 1), dtype=np.float32)
    if total:
        lp[:total] = np.concatenate([np.asarray(s, dtype=np.float32) for s in seqs if len(s)])
    return lp, lp_off


def consolidate_json_packed(blob, off, n, rel_eps: float = 0.03, abs_eps: float = 1e-6, device: int = 0, threads: int = 0,
                            flags: int = 0, logprobs=None) -> PackedResult:
    """H1g: the JSON-in / JSON-out consolidation with the JSON work on the device (kc_consolidate_json_packed).
    blob uint8 array of all candidate texts, off int64 [R*n+1]; see pack_texts().  logprobs = (lp, lp_off) from pack_logprobs():
    the likelihood-weighted vote (kc_consolidate_json_packed_weighted; records it declines keep status 1)."""
    lib = load()
    R = (len(off) - 1) // n if n else 0
    h = ctypes.c_void_p()
    if logprobs is None:
        check(lib.kc_consolidate_json_packed(blob.ctypes.data, off.ctypes.data, R, n, float(rel_eps), float(abs_eps), device, threads,
                                             flags, ctypes.byref(h)))
    else:
        import numpy as np
        lp, lp_off = logprobs
        assert lp.dtype == np.float32 and lp_off.dtype == np.int64 and len(lp_off) == len(off), "logprobs do not match the records"
        check(lib.kc_consolidate_json_packed_weighted(blob.ctypes.data, off.ctypes.data, lp.ctypes.data, lp_off.ctypes.data, R, n,
                                                      float(rel_eps), float(abs_eps), device, threads, flags, ctypes.byref(h)))
    return PackedResult(h, R)


def s32_texts_packed(n_records: int, n: int, seed: int, pinned: bool = True, threads: int = 0):
    """Schema S32 (SURVEY.md §8d) as candidate TEXTS in packed form (blob uint8, off int64 [R*n+1]), generated natively
    (kc_debug_s32_texts: exactly json.dumps' formatting; tests/test_jsongpu_host_logic.py checks that)."""
    import numpy as np
    lib = load()
    off = np.zeros(n_records * n + 1, dtype=np.int64)
    check(lib.kc_debug_s32_texts(seed, n_records, n, threads, None, 0, off.ctypes.data))
    total = int(off[-1])
    blob = pinned_empty((max(total, 1),), np.uint8) if pinned else np.empty(max(total, 1), dtype=np.uint8)
    check(lib.kc_debug_s32_texts(seed, n_records, n, threads, blob.ctypes.data, total, off.ctypes.data))
    return blob, off
