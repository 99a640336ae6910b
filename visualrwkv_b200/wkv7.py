"""WKV7 operator surface — mirrors VisualRWKV-v7/v7.00/src/model.py:45-70.

`WindBackstepping` / `RUN_CUDA_RWKV7g` keep the reference's names, argument order, assertions and
saved-tensor contract, and call the same `torch.ops.wind_backstepping.{forward,backward}` ops —
which here are implemented by the sm_100a kernels of csrc/wkv7_{fwd,bwd}.cuh through the C ABI.
"""
from __future__ import annotations

import ctypes
import os

import torch

from . import _lib

HEAD_SIZE = int(os.environ.get("RWKV_HEAD_SIZE_A", "64"))  # env contract of model.py:40
CHUNK_LEN = 16                                              # model.py:41
assert HEAD_SIZE == 64, "the sm_100a WKV7 kernels are built for head size 64 (model.py:69 hard-wires it)"


# bench.py sets PROFILE = [] to collect (kind, start_event, end_event) per launch on the current stream
PROFILE = None


def _timed(kind, fn):
    if PROFILE is None:
        return fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    PROFILE.append((kind, e0, e1))


def launch_count() -> int:
    L = _lib.lib()
    L.vrwkv_launch_count.restype = ctypes.c_ulonglong
    return int(L.vrwkv_launch_count())


BOUNDED_DECAY = 1      # include/vrwkv_b200.h: VRWKV_WKV7_BOUNDED_DECAY
CHUNK_CHECKPOINTS = 2  # VRWKV_WKV7_CHUNK_CHECKPOINTS
TF32 = 4               # VRWKV_WKV7_TF32 (round-1 kernels; outside the north-star tolerance)
CHUNK = 64


def _flags(bounded_decay, chunk_checkpoints, tf32=False):
    return ctypes.c_uint((BOUNDED_DECAY if bounded_decay else 0) | (CHUNK_CHECKPOINTS if chunk_checkpoints else 0) |
                         (TF32 if (tf32 and bounded_decay) else 0))


def cache_bytes(B: int, T: int, H: int) -> int:
    """Size of the chunk cache of forward_raw(..., chunk_cache=True): 64 KB per 64-step chunk of each (batch, head)."""
    L = _lib.lib()
    L.vrwkv_wkv7_cache_bytes.restype = ctypes.c_size_t
    return int(L.vrwkv_wkv7_cache_bytes(B, T, H))


def forward_raw(w, q, k, v, a, b, bounded_decay: bool = False, chunk_checkpoints: bool = False, tf32: bool = False,
                chunk_cache: bool = False):
    """[B,T,H,64] bf16 x6 (kernel order) -> y, s, sa through the C ABI (vrwkv_wkv7_forward_ex).

    bounded_decay=True is the caller's promise that exp(w) <= 0.607 (RWKV-7's w = -softplus(.) - 0.5, model.py:176);
    it lets the library use the chunked tensor-core kernels.  chunk_checkpoints=True (needs bounded_decay, T % 64 == 0):
    s is [B,H,T/64,64,64], one state per chunk — pass the same to backward_raw.  chunk_cache=True (needs both, not
    tf32): returns y, s, sa, cache, where cache (uint8, cache_bytes(B, T, H)) holds what the forward computed per
    chunk and the backward would otherwise recompute — pass it to backward_raw(..., cache=cache)."""
    L = _lib.lib()
    B, T, H, C = w.shape
    assert C == 64 and T % CHUNK_LEN == 0
    assert all(i.dtype == torch.bfloat16 and i.is_contiguous() and i.is_cuda for i in [w, q, k, v, a, b])
    y = torch.empty_like(v)
    chunk_checkpoints = bool(chunk_checkpoints and bounded_decay and T % CHUNK == 0)
    if chunk_cache and not (chunk_checkpoints and not tf32):
        raise ValueError("chunk_cache needs bounded_decay, chunk_checkpoints, T % 64 == 0 and not tf32")
    s = torch.empty(B, H, T // (CHUNK if chunk_checkpoints else CHUNK_LEN), C, C, dtype=torch.float32, device=w.device)
    sa = torch.empty(B, T, H, C, dtype=torch.float32, device=w.device)
    cache = torch.empty(cache_bytes(B, T, H), dtype=torch.uint8, device=w.device) if chunk_cache else None

    def run():
        with torch.cuda.device(w.device):
            if chunk_cache:
                rc = L.vrwkv_wkv7_forward_cache(B, T, H, _lib.ptr(w), _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(a),
                                                _lib.ptr(b), _lib.ptr(y), _lib.ptr(s), _lib.ptr(sa), _lib.ptr(cache),
                                                _flags(True, True), _lib.cur_stream())
            else:
                rc = L.vrwkv_wkv7_forward_ex(B, T, H, _lib.ptr(w), _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(a),
                                             _lib.ptr(b), _lib.ptr(y), _lib.ptr(s), _lib.ptr(sa), None, None,
                                             _flags(bounded_decay, chunk_checkpoints, tf32), _lib.cur_stream())
        _lib.check(rc, "vrwkv_wkv7_forward_cache" if chunk_cache else "vrwkv_wkv7_forward_ex")

    _timed("fwd", run)
    return (y, s, sa, cache) if chunk_cache else (y, s, sa)


def backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay: bool = False, tf32: bool = False, cache=None):
    """Returns dw, dq, dk, dv, da, db (bf16 [B,T,H,64]) through vrwkv_wkv7_backward_ex (the checkpoint granularity is
    read off the shape of s), or through vrwkv_wkv7_backward_cache when given the cache of forward_raw(...,
    chunk_cache=True)."""
    L = _lib.lib()
    B, T, H, C = w.shape
    chunk_checkpoints = s.shape[2] * CHUNK == T and s.shape[2] * CHUNK_LEN != T
    assert dy.dtype == torch.bfloat16 and dy.is_contiguous()
    if cache is not None:
        if not (bounded_decay and chunk_checkpoints and not tf32):
            raise ValueError("cache needs bounded_decay, 64-step checkpoints and not tf32")
        if (cache.dtype != torch.uint8 or cache.dim() != 1 or cache.numel() != cache_bytes(B, T, H)
                or not cache.is_contiguous() or cache.device != w.device):
            raise ValueError(f"cache must be a contiguous uint8 tensor of {cache_bytes(B, T, H)} bytes on {w.device}, "
                             f"got {cache.dtype} {tuple(cache.shape)} on {cache.device}")
    outs = [torch.empty_like(w) for _ in range(6)]

    def run():
        with torch.cuda.device(w.device):
            if cache is not None:
                rc = L.vrwkv_wkv7_backward_cache(B, T, H, _lib.ptr(w), _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(a),
                                                 _lib.ptr(b), _lib.ptr(dy), _lib.ptr(s), _lib.ptr(sa), _lib.ptr(cache),
                                                 *[_lib.ptr(o) for o in outs], _flags(True, True), _lib.cur_stream())
            else:
                rc = L.vrwkv_wkv7_backward_ex(B, T, H, _lib.ptr(w), _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(a),
                                              _lib.ptr(b), _lib.ptr(dy), _lib.ptr(s), _lib.ptr(sa),
                                              *[_lib.ptr(o) for o in outs],
                                              _flags(bounded_decay, chunk_checkpoints, tf32), _lib.cur_stream())
        _lib.check(rc, "vrwkv_wkv7_backward_cache" if cache is not None else "vrwkv_wkv7_backward_ex")

    _timed("bwd", run)
    return outs


def domain_check() -> None:
    """Synchronises; raises if a chunked kernel met decay outside the range promised by bounded_decay=True."""
    _lib.check(_lib.lib().vrwkv_wkv7_domain_check(), "vrwkv_wkv7_domain_check")


class WindBacksteppingBounded(torch.autograd.Function):
    """WindBackstepping for callers that build w the RWKV-7 way (exp(w) <= 0.607): chunked tensor-core kernels."""

    @staticmethod
    def forward(ctx, w, q, k, v, z, b):
        y, s, sa = forward_raw(w, q, k, v, z, b, bounded_decay=True)
        ctx.save_for_backward(w, q, k, v, z, b, s, sa)
        return y

    @staticmethod
    def backward(ctx, dy):
        w, q, k, v, z, b, s, sa = ctx.saved_tensors
        return tuple(backward_raw(w, q, k, v, z, b, dy.contiguous(), s, sa, bounded_decay=True))


class WindBackstepping(torch.autograd.Function):
    """model.py:45-65 — same ops, same allocations, same saved tensors."""

    @staticmethod
    def forward(ctx, w, q, k, v, z, b):
        _lib.load_torch_ops()
        B, T, H, C = w.shape
        assert T % CHUNK_LEN == 0
        assert all(i.dtype == torch.bfloat16 for i in [w, q, k, v, z, b])
        assert all(i.is_contiguous() for i in [w, q, k, v, z, b])
        y = torch.empty_like(v)
        s = torch.empty(B, H, T // CHUNK_LEN, C, C, dtype=torch.float32, device=w.device)
        sa = torch.empty(B, T, H, C, dtype=torch.float32, device=w.device)
        _timed("fwd", lambda: torch.ops.wind_backstepping.forward(w, q, k, v, z, b, y, s, sa))
        ctx.save_for_backward(w, q, k, v, z, b, s, sa)
        return y

    @staticmethod
    def backward(ctx, dy):
        assert all(i.dtype == torch.bfloat16 for i in [dy])
        dy = dy.contiguous()  # the reference asserts; autograd may hand us a strided view
        w, q, k, v, z, b, s, sa = ctx.saved_tensors
        dw, dq, dk, dv, dz, db = [torch.empty_like(x) for x in [w, q, k, v, z, b]]
        _timed("bwd", lambda: torch.ops.wind_backstepping.backward(w, q, k, v, z, b, dy, s, sa, dw, dq, dk, dv, dz, db))
        return dw, dq, dk, dv, dz, db


def RUN_CUDA_RWKV7g(q, w, k, v, a, b, bounded_decay: bool = False):
    """model.py:67-70: six [B,T,H*64] bf16 -> [B,T,H*64] bf16, differentiable in all six.

    bounded_decay=True (not in the reference signature): w was built as -softplus(.) - 0.5, see forward_raw."""
    B, T, HC = q.shape
    q, w, k, v, a, b = [i.view(B, T, HC // 64, 64) for i in [q, w, k, v, a, b]]
    fn = WindBacksteppingBounded if bounded_decay else WindBackstepping
    return fn.apply(w, q, k, v, a, b).view(B, T, HC)


def wkv7_forward_state(w, q, k, v, a, b, state_in=None, want_checkpoints: bool = False, bounded_decay: bool = False,
                       state_out=None):
    """Stateful forward (SURVEY.md §8f-2): returns (y, state_out[, s, sa]); inference only (no grad).

    state_in / state_out: f32 [B,H,64,64] (S_ij row-major).  T need not be a multiple of 16 unless
    checkpoints are requested.  bounded_decay=True (the caller's promise exp(w) <= 0.607, see forward_raw) lets a
    prefill whose T is a multiple of 64 run on the chunked tensor-core kernel; any other T (the T = 1 decode step
    included) runs on the step-by-step kernel either way.  state_out may be given (and, for T % 64 != 0, may be state_in
    itself: the step-by-step kernel reads a head's state once at the start and writes it once at the end).
    """
    L = _lib.lib()
    B, T, H, C = w.shape
    assert C == 64 and all(i.dtype == torch.bfloat16 and i.is_contiguous() and i.is_cuda for i in [w, q, k, v, a, b])
    y = torch.empty_like(v)
    if state_out is None:
        state_out = torch.empty(B, H, C, C, dtype=torch.float32, device=w.device)
    assert state_out.dtype == torch.float32 and state_out.is_contiguous() and state_out.shape == (B, H, C, C)
    assert state_out is not state_in or T % CHUNK != 0 or not bounded_decay, "in-place state only on the step-by-step kernel"
    s = sa = None
    if want_checkpoints:
        s = torch.empty(B, H, T // CHUNK_LEN, C, C, dtype=torch.float32, device=w.device)
        sa = torch.empty(B, T, H, C, dtype=torch.float32, device=w.device)
    if state_in is not None:
        assert state_in.dtype == torch.float32 and state_in.is_contiguous() and state_in.shape == (B, H, C, C)
    with torch.cuda.device(w.device):
        rc = L.vrwkv_wkv7_forward_ex(B, T, H, _lib.ptr(w), _lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(a),
                                     _lib.ptr(b), _lib.ptr(y), _lib.ptr(s), _lib.ptr(sa), _lib.ptr(state_in),
                                     _lib.ptr(state_out), _flags(bool(bounded_decay and T % CHUNK == 0), False, False),
                                     _lib.cur_stream())
    _lib.check(rc, "vrwkv_wkv7_forward_ex")
    return (y, state_out, s, sa) if want_checkpoints else (y, state_out)


def set_variant(fwd: int = 0, bwd: int = 0) -> None:
    _lib.check(_lib.lib().vrwkv_wkv7_set_variant(ctypes.c_int(fwd), ctypes.c_int(bwd)), "set_variant")
