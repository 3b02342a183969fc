"""ctypes binding of libkvpress_b200.so (the C ABI in include/kvpress_b200.h).

torch is used here only as the owner of device memory and streams: tensors are handed to the
library as raw pointers + element strides, outputs and scratch are allocated with torch's caching
allocator, kernels are enqueued on torch's current stream. There is NO fallback: if the shared
library is missing or a tensor is not a CUDA tensor, calls raise.
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path
from typing import Optional

import torch

_LIB_NAME = "libkvpress_b200.so"
_LIB_PATH = Path(__file__).resolve().parent / _LIB_NAME

SCORER_GENERIC, SCORER_KNORM, SCORER_STREAMING, SCORER_SNAPKV, SCORER_EXPECTED_ATTENTION, SCORER_KEYDIFF = range(6)
_DTYPES = {torch.bfloat16: 0, torch.float16: 1}


class KvpProblem(ctypes.Structure):
    """Mirror of `struct kvp_problem`."""

    _fields_ = [
        ("B", ctypes.c_int32),
        ("Hkv", ctypes.c_int32),
        ("Hq", ctypes.c_int32),
        ("S", ctypes.c_int32),
        ("D", ctypes.c_int32),
        ("n_kept", ctypes.c_int32),
        ("dtype", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("k_stride", ctypes.c_int64 * 3),
        ("v_stride", ctypes.c_int64 * 3),
    ]


class NativeLibraryError(RuntimeError):
    pass


# name -> (restype, argtypes); every symbol include/kvpress_b200.h declares
_P = ctypes.c_void_p
_PP = ctypes.POINTER(KvpProblem)
_SZ = ctypes.c_size_t
_I = ctypes.c_int32
SIGNATURES = {
    "kvp_abi_version": (ctypes.c_int, []),
    "kvp_status_string": (ctypes.c_char_p, [ctypes.c_int]),
    "kvp_last_cuda_error": (ctypes.c_char_p, []),
    "kvp_workspace_bytes": (ctypes.c_int, [_PP, ctypes.c_int, ctypes.POINTER(_SZ)]),
    "kvp_launches_per_compress": (ctypes.c_int, [_PP, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "kvp_workspace_check": (ctypes.c_int, [_PP, ctypes.c_int, _P, _SZ, _P]),
    "kvp_knorm_score": (ctypes.c_int, [_PP, _P, _P, _P]),
    "kvp_knorm_compress": (ctypes.c_int, [_PP, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "kvp_streaming_score": (ctypes.c_int, [_PP, _I, _P, _P]),
    "kvp_streaming_compress": (ctypes.c_int, [_PP, _I, _P, _P, _P, _P, _P, _P]),
    "kvp_snapkv_score": (ctypes.c_int, [_PP, _P, _P, _I, _I, _P, _P, _SZ, _P]),
    "kvp_snapkv_compress": (ctypes.c_int, [_PP, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    "kvp_expected_attention_score": (
        ctypes.c_int, [_PP, _P, _P, _P, _P, ctypes.c_float, _I, _I, _P, _P, _SZ, _P]),
    "kvp_expected_attention_compress": (
        ctypes.c_int, [_PP, _P, _P, _P, _P, ctypes.c_float, _I, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    "kvp_scores_compress": (
        ctypes.c_int, [_PP, _P, ctypes.POINTER(ctypes.c_int64), _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "kvp_keydiff_score": (ctypes.c_int, [_PP, _P, _P, _P, _SZ, _P]),
    "kvp_keydiff_compress": (ctypes.c_int, [_PP, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "kvp_scores_select": (ctypes.c_int, [_PP, _P, ctypes.POINTER(ctypes.c_int64), _P, _P, _SZ, _P]),
    "kvp_scores_compress_rerotate": (
        ctypes.c_int, [_PP, _P, ctypes.POINTER(ctypes.c_int64), _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
}

_lib: Optional[ctypes.CDLL] = None


def library_path() -> Path:
    return Path(os.environ.get("KVPRESS_B200_LIB", _LIB_PATH))


def load() -> ctypes.CDLL:
    """Load the shared library (once) and bind every declared symbol. Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not path.exists():
        raise NativeLibraryError(
            f"{path} not found: build it with `python -m kvpress_b200.build` (needs nvcc). "
            "kvpress_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(str(path))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.kvp_abi_version() != 1:
        raise NativeLibraryError(f"ABI version mismatch: library reports {lib.kvp_abi_version()}")
    _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        lib = load()
        msg = lib.kvp_status_string(rc).decode()
        if rc == -6:
            msg += ": " + lib.kvp_last_cuda_error().decode()
        raise RuntimeError(f"{what} failed: {msg} (status {rc})")


def _pinned_ok(t: torch.Tensor) -> bool:
    """A pinned host tensor is addressable from the device (UVA): kernels may gather its rows over PCIe."""
    return (not t.is_cuda) and t.is_pinned() and torch.cuda.is_available()


def _require_cuda_kv(keys: torch.Tensor, values: torch.Tensor, pinned_values: bool = False,
                     pinned_keys: bool = False) -> None:
    k_ok = keys.is_cuda or (pinned_keys and _pinned_ok(keys))
    v_ok = values.is_cuda or (pinned_values and _pinned_ok(values))
    if not (k_ok and v_ok):
        raise RuntimeError(
            "kvpress_b200 runs on CUDA tensors only (sm_100a kernels); got "
            f"keys on {keys.device}, values on {values.device}. There is no CPU path."
        )
    if keys.dtype not in _DTYPES or values.dtype != keys.dtype:
        raise RuntimeError(f"kvpress_b200 supports bf16/fp16 caches, got {keys.dtype}/{values.dtype}")
    if keys.dim() != 4 or values.shape != keys.shape:
        raise RuntimeError(f"expected K, V of shape [B, Hkv, S, D], got {tuple(keys.shape)}, {tuple(values.shape)}")


def _out_device(keys: torch.Tensor) -> torch.device:
    return keys.device if keys.is_cuda else torch.device("cuda", torch.cuda.current_device())


def _rows_ok(t: torch.Tensor) -> bool:
    if t.stride(3) != 1 or t.data_ptr() % 16:
        return False
    for dim in range(3):
        if t.shape[dim] > 1 and (t.stride(dim) % 8 or t.stride(dim) < 0):
            return False
    return t.shape[2] == 1 or t.stride(2) >= t.shape[3]


def _normalise(t: torch.Tensor) -> torch.Tensor:
    """Strided views are consumed as they are; only layouts the kernels cannot address are copied."""
    if _rows_ok(t):
        return t
    if not t.is_cuda:
        raise RuntimeError("a pinned host K/V view must already have 16-byte aligned, unit-stride rows")
    return t.contiguous()


def _strides(t: torch.Tensor):
    return tuple(int(t.stride(d)) if t.shape[d] > 1 else 0 for d in range(3))


_PROBLEMS: dict = {}


def make_problem(keys: torch.Tensor, values: torch.Tensor, n_kept: int, num_q_heads: Optional[int] = None) -> KvpProblem:
    """kvp_problem of one call. Structs are cached per (shape, strides, n_kept, Hq, dtype) and must be treated
    as read-only by callers: DecodingPress / per-layer hooks repeat the same few problems thousands of times."""
    key = (keys.shape, keys.stride(), values.stride(), int(n_kept), num_q_heads, keys.dtype)
    p = _PROBLEMS.get(key)
    if p is None:
        p = _build_problem(keys, values, n_kept, num_q_heads)
        if len(_PROBLEMS) > 1024:
            _PROBLEMS.clear()
        _PROBLEMS[key] = p
    return p


def _build_problem(keys: torch.Tensor, values: torch.Tensor, n_kept: int, num_q_heads: Optional[int] = None) -> KvpProblem:
    B, H, S, D = keys.shape
    p = KvpProblem()
    p.B, p.Hkv, p.S, p.D = B, H, S, D
    p.Hq = int(num_q_heads) if num_q_heads else H
    p.n_kept = int(n_kept)
    p.dtype = _DTYPES[keys.dtype]
    ks, vs = _strides(keys), _strides(values)
    # a row stride of 0 only happens for S == 1; keep it addressable
    p.k_stride = (ctypes.c_int64 * 3)(ks[0], ks[1], ks[2] if S > 1 else D)
    p.v_stride = (ctypes.c_int64 * 3)(vs[0], vs[1], vs[2] if S > 1 else D)
    return p


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device, as an integer handle."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> int:
    """Raw address (0 = NULL); ctypes converts ints to void* through the declared argtypes."""
    return 0 if t is None else t.data_ptr()


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def _guard(device: torch.device):
    """Device guard only when the tensor's device is not the current one (the common per-layer hook call
    skips the set-device round trip)."""
    if device.type != "cuda" or device.index is None or device.index == torch.cuda.current_device():
        return _NO_GUARD
    return torch.cuda.device(device)


_WS_BYTES: dict = {}


def workspace_bytes(p: KvpProblem, scorer: int) -> int:
    """kvp_workspace_bytes, asked once per (shape, scorer)."""
    key = (p.B, p.Hkv, p.Hq, p.S, p.D, p.dtype, scorer)
    n = _WS_BYTES.get(key)
    if n is None:
        out = _SZ(0)
        _check(load().kvp_workspace_bytes(ctypes.byref(p), scorer, ctypes.byref(out)), "kvp_workspace_bytes")
        n = _WS_BYTES[key] = int(out.value)
        if len(_WS_BYTES) > 4096:
            _WS_BYTES.clear()
    return n


def launches_per_compress(p: KvpProblem, scorer: int) -> int:
    out = ctypes.c_int(0)
    _check(load().kvp_launches_per_compress(ctypes.byref(p), scorer, ctypes.byref(out)), "kvp_launches_per_compress")
    return int(out.value)


def _alloc_out(keys: torch.Tensor, n_kept: int, want_idx: bool, want_scores: bool):
    B, H, S, D = keys.shape
    dev = _out_device(keys)
    k_out = torch.empty((B, H, n_kept, D), dtype=keys.dtype, device=dev)
    v_out = torch.empty_like(k_out)
    idx = torch.empty((B, H, n_kept), dtype=torch.int32, device=dev) if want_idx else None
    scores = torch.empty((B, H, S), dtype=keys.dtype, device=dev) if want_scores else None
    return k_out, v_out, idx, scores


_WS_CACHE: dict = {}


def _workspace(p: KvpProblem, scorer: int, device) -> torch.Tensor:
    """Scratch for one call. Calls on one stream execute in order, so one grow-only buffer per (device, stream)
    is reused instead of allocated per call; under CUDA-graph capture a fresh buffer from the graph's pool is
    used (it must live exactly as long as the graph)."""
    need = workspace_bytes(p, scorer)
    if device.type != "cuda":
        return torch.empty(need, dtype=torch.uint8, device=device)
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(need, dtype=torch.uint8, device=device)
    key = (device.index, _stream())
    ws = _WS_CACHE.get(key)
    if ws is None or ws.numel() < need:
        if len(_WS_CACHE) > 64:
            _WS_CACHE.clear()
        ws = _WS_CACHE[key] = torch.empty(max(need, 1 << 20), dtype=torch.uint8, device=device)
    return ws


# --------------------------------------------------------------------------------------------------
# captured calls: one compress call bound to fixed tensors, replayed as ONE graph launch
# --------------------------------------------------------------------------------------------------
class GraphedCall:
    """`fn()` (any sequence of native.* calls on fixed input tensors) captured into a CUDA graph.

    The C-ABI calls only enqueue kernels / memset nodes on the current stream (the ExpectedAttention side
    stream forks from and joins back into it), never synchronise and never allocate, so they are capturable
    as they are. `replay()` costs one cudaGraphLaunch on the host instead of 1-7 launches + their argument
    marshalling: it makes the call GPU-bound on any host (DecodingPress compactions, repeated same-shape
    prefill layers, bench.py). Outputs are the tensors `fn` returned; they are overwritten by every replay.
    The inputs must stay alive and at the same addresses (update them in place)."""

    def __init__(self, fn, warmup: int = 2):
        if not torch.cuda.is_available():
            raise RuntimeError("GraphedCall needs a CUDA device")
        self._fn = fn
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # warm-up off the capture: lazy inits (func attributes, side stream, ...)
            for _ in range(max(1, warmup)):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.outputs = fn()

    def replay(self):
        self.graph.replay()
        return self.outputs

    __call__ = replay


def capture(fn, warmup: int = 2) -> GraphedCall:
    return GraphedCall(fn, warmup)


def workspace_check(p: KvpProblem, scorer: int, workspace: torch.Tensor) -> None:
    """Raises if a kernel of the last call on this workspace abandoned a bounded wait (kvp_workspace_check;
    synchronises the current stream). Debugging aid: the wait only expires on a library bug."""
    _check(load().kvp_workspace_check(ctypes.byref(p), scorer, _ptr(workspace), workspace.numel(), _stream()),
           "kvp_workspace_check")


# --------------------------------------------------------------------------------------------------
# Knorm
# --------------------------------------------------------------------------------------------------
def knorm_score(keys: torch.Tensor) -> torch.Tensor:
    _require_cuda_kv(keys, keys)
    keys = _normalise(keys)
    p = make_problem(keys, keys, 0)
    scores = torch.empty(keys.shape[:3], dtype=keys.dtype, device=keys.device)
    with _guard(keys.device):
        _check(load().kvp_knorm_score(ctypes.byref(p), _ptr(keys), _ptr(scores), _stream()), "kvp_knorm_score")
    return scores


def knorm_compress(keys, values, n_kept: int, return_indices: bool = False, return_scores: bool = False,
                   _pinned_values: bool = False):
    _require_cuda_kv(keys, values, pinned_values=_pinned_values)
    keys, values = _normalise(keys), _normalise(values)
    p = make_problem(keys, values, n_kept)
    k_out, v_out, idx, scores = _alloc_out(keys, n_kept, return_indices, return_scores)
    if n_kept > 0:
        with _guard(keys.device):
            ws = _workspace(p, SCORER_KNORM, keys.device)
            _check(
                load().kvp_knorm_compress(
                    ctypes.byref(p), _ptr(keys), _ptr(values), _ptr(k_out), _ptr(v_out), _ptr(idx), _ptr(scores),
                    _ptr(ws), ws.numel(), _stream()),
                "kvp_knorm_compress",
            )
    return k_out, v_out, idx, scores


# --------------------------------------------------------------------------------------------------
# KeyDiff
# --------------------------------------------------------------------------------------------------
def keydiff_score(keys: torch.Tensor) -> torch.Tensor:
    _require_cuda_kv(keys, keys)
    keys = _normalise(keys)
    p = make_problem(keys, keys, 0)
    scores = torch.empty(keys.shape[:3], dtype=keys.dtype, device=keys.device)
    with _guard(keys.device):
        ws = _workspace(p, SCORER_KEYDIFF, keys.device)
        _check(load().kvp_keydiff_score(ctypes.byref(p), _ptr(keys), _ptr(scores), _ptr(ws), ws.numel(), _stream()),
               "kvp_keydiff_score")
    return scores


def keydiff_compress(keys, values, n_kept: int, return_indices: bool = False, return_scores: bool = False,
                     _pinned_values: bool = False):
    _require_cuda_kv(keys, values, pinned_values=_pinned_values)
    keys, values = _normalise(keys), _normalise(values)
    p = make_problem(keys, values, n_kept)
    k_out, v_out, idx, scores = _alloc_out(keys, n_kept, return_indices, return_scores)
    if n_kept > 0:
        with _guard(keys.device):
            ws = _workspace(p, SCORER_KEYDIFF, keys.device)
            _check(
                load().kvp_keydiff_compress(
                    ctypes.byref(p), _ptr(keys), _ptr(values), _ptr(k_out), _ptr(v_out), _ptr(idx), _ptr(scores),
                    _ptr(ws), ws.numel(), _stream()),
                "kvp_keydiff_compress",
            )
    return k_out, v_out, idx, scores


# --------------------------------------------------------------------------------------------------
# StreamingLLM
# --------------------------------------------------------------------------------------------------
def streaming_score(keys: torch.Tensor, n_kept: int, n_sink: int) -> torch.Tensor:
    _require_cuda_kv(keys, keys)
    p = make_problem(keys, keys, n_kept)
    scores = torch.empty(keys.shape[:3], dtype=keys.dtype, device=keys.device)
    with _guard(keys.device):
        _check(load().kvp_streaming_score(ctypes.byref(p), n_sink, _ptr(scores), _stream()), "kvp_streaming_score")
    return scores


def streaming_compress(keys, values, n_kept: int, n_sink: int, return_indices: bool = False,
                       _pinned_kv: bool = False):
    _require_cuda_kv(keys, values, pinned_values=_pinned_kv, pinned_keys=_pinned_kv)
    keys, values = _normalise(keys), _normalise(values)
    p = make_problem(keys, values, n_kept)
    k_out, v_out, idx, _ = _alloc_out(keys, n_kept, return_indices, False)
    if n_kept > 0:
        with _guard(k_out.device):
            _check(
                load().kvp_streaming_compress(
                    ctypes.byref(p), n_sink, _ptr(keys), _ptr(values), _ptr(k_out), _ptr(v_out), _ptr(idx), _stream()),
                "kvp_streaming_compress",
            )
    return k_out, v_out, idx


# --------------------------------------------------------------------------------------------------
# SnapKV
# --------------------------------------------------------------------------------------------------
def _check_q(q_window: torch.Tensor, keys: torch.Tensor, window: int):
    B, _, _, D = keys.shape
    if q_window.dim() != 4 or q_window.shape[0] != B or q_window.shape[2] != window or q_window.shape[3] != D:
        raise RuntimeError(f"q_window must be [B, Hq, {window}, {D}], got {tuple(q_window.shape)}")
    if q_window.dtype != keys.dtype or q_window.device != keys.device:
        raise RuntimeError("q_window must share dtype and device with the keys")
    return q_window.contiguous()


def snapkv_score(keys, q_window, window: int, kernel_size: int) -> torch.Tensor:
    _require_cuda_kv(keys, keys)
    keys = _normalise(keys)
    q_window = _check_q(q_window, keys, window)
    p = make_problem(keys, keys, 0, q_window.shape[1])
    scores = torch.empty(keys.shape[:3], dtype=keys.dtype, device=keys.device)
    with _guard(keys.device):
        ws = _workspace(p, SCORER_SNAPKV, keys.device)
        _check(
            load().kvp_snapkv_score(
                ctypes.byref(p), _ptr(keys), _ptr(q_window), window, kernel_size, _ptr(scores), _ptr(ws), ws.numel(),
                _stream()),
            "kvp_snapkv_score",
        )
    return scores


def snapkv_compress(keys, values, q_window, window: int, kernel_size: int, n_kept: int,
                    return_indices: bool = False, return_scores: bool = False, _pinned_values: bool = False):
    _require_cuda_kv(keys, values, pinned_values=_pinned_values)
    keys, values = _normalise(keys), _normalise(values)
    q_window = _check_q(q_window, keys, window)
    p = make_problem(keys, values, n_kept, q_window.shape[1])
    k_out, v_out, idx, scores = _alloc_out(keys, n_kept, return_indices, return_scores)
    if n_kept > 0:
        with _guard(keys.device):
            ws = _workspace(p, SCORER_SNAPKV, keys.device)
            _check(
                load().kvp_snapkv_compress(
                    ctypes.byref(p), _ptr(keys), _ptr(values), _ptr(q_window), window, kernel_size, _ptr(k_out),
                    _ptr(v_out), _ptr(idx), _ptr(scores), _ptr(ws), ws.numel(), _stream()),
                "kvp_snapkv_compress",
            )
    return k_out, v_out, idx, scores


# --------------------------------------------------------------------------------------------------
# ExpectedAttention
# --------------------------------------------------------------------------------------------------
def _check_stats(mu, cov, keys):
    B, _, _, D = keys.shape
    if mu.dim() != 3 or mu.shape[0] != B or mu.shape[2] != D:
        raise RuntimeError(f"mu must be [B, Hq, {D}], got {tuple(mu.shape)}")
    mu = mu.to(keys.dtype).contiguous()
    if cov is not None:
        if tuple(cov.shape) != (B, mu.shape[1], D, D):
            raise RuntimeError(f"cov must be [B, Hq, {D}, {D}], got {tuple(cov.shape)}")
        cov = cov.to(keys.dtype).contiguous()
    return mu, cov


def expected_attention_score(keys, values, mu, cov, epsilon: float, n_sink: int, use_vnorm: bool) -> torch.Tensor:
    _require_cuda_kv(keys, values)
    keys, values = _normalise(keys), _normalise(values)
    mu, cov = _check_stats(mu, cov, keys)
    p = make_problem(keys, values, 0, mu.shape[1])
    scores = torch.empty(keys.shape[:3], dtype=keys.dtype, device=keys.device)
    with _guard(keys.device):
        ws = _workspace(p, SCORER_EXPECTED_ATTENTION, keys.device)
        _check(
            load().kvp_expected_attention_score(
                ctypes.byref(p), _ptr(keys), _ptr(values), _ptr(mu), _ptr(cov), float(epsilon), n_sink,
                int(bool(use_vnorm)), _ptr(scores), _ptr(ws), ws.numel(), _stream()),
            "kvp_expected_attention_score",
        )
    return scores


def expected_attention_compress(keys, values, mu, cov, epsilon: float, n_sink: int, use_vnorm: bool, n_kept: int,
                                return_indices: bool = False, return_scores: bool = False):
    _require_cuda_kv(keys, values)
    keys, values = _normalise(keys), _normalise(values)
    mu, cov = _check_stats(mu, cov, keys)
    p = make_problem(keys, values, n_kept, mu.shape[1])
    k_out, v_out, idx, scores = _alloc_out(keys, n_kept, return_indices, return_scores)
    if n_kept > 0:
        with _guard(keys.device):
            ws = _workspace(p, SCORER_EXPECTED_ATTENTION, keys.device)
            _check(
                load().kvp_expected_attention_compress(
                    ctypes.byref(p), _ptr(keys), _ptr(values), _ptr(mu), _ptr(cov), float(epsilon), n_sink,
                    int(bool(use_vnorm)), _ptr(k_out), _ptr(v_out), _ptr(idx), _ptr(scores), _ptr(ws), ws.numel(),
                    _stream()),
                "kvp_expected_attention_compress",
            )
    return k_out, v_out, idx, scores


# --------------------------------------------------------------------------------------------------
# generic scores (wrapper presses, user-defined ScorerPress subclasses)
# --------------------------------------------------------------------------------------------------
def scores_compress(scores: torch.Tensor, keys, values, n_kept: int, return_indices: bool = False):
    """Top-k + compaction for caller-supplied scores [B, Hkv, S] (wrapper presses, user ScorerPress subclasses).

    The selection kernels rank 16-bit keys: scores are compared IN THE CACHE DTYPE. The in-scope scorers return that
    dtype already (as the reference's do); fp32 scores of a custom press are rounded to it first, so values that
    differ only below bf16 / fp16 resolution become ties and go to the lowest positions, where the reference's fp32
    `topk` would still order them."""
    _require_cuda_kv(keys, values)
    keys, values = _normalise(keys), _normalise(values)
    if tuple(scores.shape) != tuple(keys.shape[:3]) or scores.device != keys.device:
        raise RuntimeError(f"scores must be [B, Hkv, S] on the cache device, got {tuple(scores.shape)}")
    scores = scores.to(keys.dtype)
    if scores.stride(2) != 1:
        scores = scores.contiguous()
    p = make_problem(keys, values, n_kept)
    k_out, v_out, idx, _ = _alloc_out(keys, n_kept, return_indices, False)
    if n_kept > 0:
        sstride = (ctypes.c_int64 * 2)(
            scores.stride(0) if scores.shape[0] > 1 else 0, scores.stride(1) if scores.shape[1] > 1 else 0)
        with _guard(keys.device):
            ws = _workspace(p, SCORER_GENERIC, keys.device)
            _check(
                load().kvp_scores_compress(
                    ctypes.byref(p), _ptr(scores), sstride, _ptr(keys), _ptr(values), _ptr(k_out), _ptr(v_out),
                    _ptr(idx), _ptr(ws), ws.numel(), _stream()),
                "kvp_scores_compress",
            )
    return k_out, v_out, idx


def scores_select(scores: torch.Tensor, n_kept: int) -> torch.Tensor:
    """Positions of the n_kept largest scores of every row of a [B, H, S] bf16/fp16 CUDA tensor, ascending
    (ties to the lowest positions), int32 [B, H, n_kept]. No K/V involved."""
    if not scores.is_cuda or scores.dtype not in _DTYPES or scores.dim() != 3:
        raise RuntimeError(f"scores must be a CUDA bf16/fp16 [B, H, S] tensor, got {scores.dtype} on {scores.device}")
    if scores.stride(2) != 1:
        scores = scores.contiguous()
    B, H, S = scores.shape
    p = KvpProblem()
    p.B, p.Hkv, p.Hq, p.S, p.D, p.n_kept, p.dtype = B, H, H, S, 8, int(n_kept), _DTYPES[scores.dtype]
    idx = torch.empty((B, H, n_kept), dtype=torch.int32, device=scores.device)
    if n_kept > 0:
        sstride = (ctypes.c_int64 * 2)(scores.stride(0) if B > 1 else 0, scores.stride(1) if H > 1 else 0)
        with _guard(scores.device):
            ws = _workspace(p, SCORER_GENERIC, scores.device)
            _check(load().kvp_scores_select(ctypes.byref(p), _ptr(scores), sstride, _ptr(idx), _ptr(ws), ws.numel(),
                                            _stream()), "kvp_scores_select")
    return idx


def scores_compress_rerotate(scores: torch.Tensor, keys, values, n_kept: int, inv_freq: torch.Tensor,
                             return_indices: bool = False):
    """KeyRerotationPress: top-k + compaction with the kept keys re-rotated to their new positions."""
    _require_cuda_kv(keys, values)
    keys, values = _normalise(keys), _normalise(values)
    if tuple(scores.shape) != tuple(keys.shape[:3]) or scores.device != keys.device:
        raise RuntimeError(f"scores must be [B, Hkv, S] on the cache device, got {tuple(scores.shape)}")
    if inv_freq.numel() * 2 != keys.shape[3]:
        raise RuntimeError(f"inv_freq must have head_dim/2 = {keys.shape[3] // 2} entries, got {inv_freq.numel()}")
    scores = scores.to(keys.dtype)
    if scores.stride(2) != 1:
        scores = scores.contiguous()
    inv_freq = inv_freq.to(device=keys.device, dtype=torch.float32).contiguous()
    p = make_problem(keys, values, n_kept)
    k_out, v_out, idx, _ = _alloc_out(keys, n_kept, return_indices, False)
    if n_kept > 0:
        sstride = (ctypes.c_int64 * 2)(
            scores.stride(0) if scores.shape[0] > 1 else 0, scores.stride(1) if scores.shape[1] > 1 else 0)
        with _guard(keys.device):
            ws = _workspace(p, SCORER_GENERIC, keys.device)
            _check(
                load().kvp_scores_compress_rerotate(
                    ctypes.byref(p), _ptr(scores), sstride, _ptr(keys), _ptr(values), _ptr(inv_freq), _ptr(k_out),
                    _ptr(v_out), _ptr(idx), _ptr(ws), ws.numel(), _stream()),
                "kvp_scores_compress_rerotate",
            )
    return k_out, v_out, idx
