"""GPU tests of the WKV7 chunk cache: the x6 forward writes each chunk's masked matrices A_qb, A_qk, A_ak and its
triangular inverse (I - A_ab)^-1 (parts 0 and 1 of the bf16 split), and the x3 backward loads them instead of
recomputing them.  Held to the bounds of the uncached chunked path (tests/test_wkv7_gpu.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import wkv7 as O
from oracle import wkv7_chunked as OC

pytestmark = pytest.mark.gpu
REF_ERRORS = os.path.join(os.path.dirname(__file__), "golden", "wkv7_refkernel_errors_b2t512h4.npz")
NAMES = ["dw", "dq", "dk", "dv", "da", "db"]
TILE = 8192


def run_cached(inp):
    from visualrwkv_b200 import wkv7 as W
    w, q, k, v, a, b, dy = inp
    y, s, sa, cache = W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True, chunk_cache=True)
    g = W.backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay=True, cache=cache)
    torch.cuda.synchronize()
    W.domain_check()
    return y, s, sa, cache, g


def run_uncached(inp):
    from visualrwkv_b200 import wkv7 as W
    w, q, k, v, a, b, dy = inp
    out = W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True)
    assert len(out) == 3
    y, s, sa = out
    g = W.backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay=True)
    torch.cuda.synchronize()
    W.domain_check()
    return y, s, sa, g


@pytest.mark.parametrize("shape,kind,seed", [((2, 64, 3), "realistic", 7), ((1, 64, 1), "realistic", 3), ((3, 256, 5), "realistic", 2),
                                               ((2, 512, 3), "realistic", 5), ((1, 2048, 2), "realistic", 6),
                                               ((2, 256, 2), "stress", 8), ((1, 1024, 2), "stress", 4)])
def test_cached_gradients_vs_fp64_oracle(shape, kind, seed):
    B, T, H = shape
    cpu = O.make_inputs(B, T, H, 64, seed=seed, kind=kind)
    inp = [x.cuda() for x in cpu]
    y, s, sa, _, g = run_cached(inp)
    y0, s0, sa0, _ = run_uncached(inp)
    # writing the cache does not change what the forward computes
    assert torch.equal(y, y0) and torch.equal(s, s0) and torch.equal(sa, sa0)
    y64, s64, sa64 = O.forward(*cpu[:6])
    g64 = O.backward(*cpu, s64, sa64)
    for n, x, r in zip(NAMES, g, g64):
        assert O.err_ratio(x.float().cpu().numpy(), r) < 2.0e-3, n


def test_cached_not_worse_than_reference_kernel():
    z = np.load(REF_ERRORS)
    cpu = O.make_inputs(int(z["B"]), int(z["T"]), int(z["H"]), 64, seed=int(z["seed"]), kind=str(z["kind"]))
    _, _, _, _, g = run_cached([x.cuda() for x in cpu])
    y64, s64, sa64 = O.forward(*cpu[:6])
    g64 = O.backward(*cpu, s64, sa64)
    for n, x, t in zip(NAMES, g, g64):
        assert O.err_ratio(x.float().cpu().numpy(), t) <= 1.02 * float(z[n]), n


def decode_pair(cache, item, tile0, tile1):
    """Tiles `tile0` + `tile1` of an item (two bf16 parts, [t][s], 128-byte rows with 16-byte chunks XOR-swizzled by
    t & 7) -> fp64 [64, 64]."""
    t = torch.arange(64).view(64, 1)
    s = torch.arange(64).view(1, 64)
    elem = (t * 128 + (((s >> 3) ^ (t & 7)) << 4) + (s & 7) * 2) // 2
    base = item * 8 * TILE
    out = torch.zeros(64, 64, dtype=torch.float64)
    for tile in (tile0, tile1):
        raw = cache[base + tile * TILE: base + (tile + 1) * TILE].view(torch.bfloat16).float().double()
        out += raw[elem.reshape(-1)].view(64, 64)
    return out


def test_cache_tiles_match_the_chunk_oracle():
    """The layout the backward relies on: item c*B*H + b*H + h holds A_qb, A_qk, A_ak and (I - A_ab)^-1 of chunk c of
    (b, h), part 0 + part 1 equal to the fp64 chunk matrices to the accuracy of a two-part bf16 split."""
    B, T, H = 2, 128, 2
    cpu = O.make_inputs(B, T, H, 64, seed=13)
    _, _, _, cache, _ = run_cached([x.cuda() for x in cpu])
    cache = cache.cpu()
    *_, inter = OC.chunk_forward(*cpu[:6], want=True)
    eye = torch.eye(64, dtype=torch.float64)
    for c, m in enumerate(inter):
        for bb in range(B):
            for hh in range(H):
                item = c * B * H + bb * H + hh
                ref = {"qb": m["A_qb"][bb, hh], "qk": m["A_qk"][bb, hh], "ak": m["A_ak"][bb, hh],
                       "tinv": torch.linalg.inv(eye - m["A_ab"][bb, hh])}
                got = {"qb": decode_pair(cache, item, 0, 2), "qk": decode_pair(cache, item, 1, 3),
                       "ak": decode_pair(cache, item, 4, 5), "tinv": decode_pair(cache, item, 6, 7)}
                for n in ref:
                    r, x = ref[n], got[n]
                    assert torch.equal(x.triu(1 if n != "ak" else 0), torch.zeros_like(x)), (n, c, bb, hh)
                    err = float((x - r).abs().max() / r.abs().max())
                    assert err < 1e-4, (n, c, bb, hh, err)


def test_cfg2_size_cached_backward_agrees_with_uncached():
    """BASELINE cfg2 size (B8 T2048 H12: about 20 items per CTA, the flag-chained dS hand-off under load)."""
    inp = [x.cuda() for x in O.make_inputs(8, 2048, 12, 64, seed=42)]
    y, s, sa, cache, g = run_cached(inp)
    y0, s0, sa0, g0 = run_uncached(inp)
    assert torch.equal(y, y0) and torch.equal(s, s0) and torch.equal(sa, sa0)
    for n, x, r in zip(NAMES, g, g0):
        assert torch.isfinite(x.float()).all(), n
        assert O.err_ratio(x.float().cpu().numpy(), r.float().cpu().numpy().astype(np.float64)) < 1e-3, n


def test_wrong_cache_is_rejected():
    from visualrwkv_b200 import wkv7 as W
    w, q, k, v, a, b, dy = [x.cuda() for x in O.make_inputs(1, 128, 2, 64, seed=3)]
    y, s, sa, cache = W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True, chunk_cache=True)
    assert cache.numel() == W.cache_bytes(1, 128, 2) == 2 * 2 * 64 * 1024
    for bad in (cache[:-1024], torch.zeros(cache.numel() + 1024, dtype=torch.uint8, device="cuda"),
                cache.view(torch.int32), cache.view(2, -1), cache.cpu()):
        with pytest.raises(ValueError):
            W.backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay=True, cache=bad)
    with pytest.raises(ValueError):   # the cache needs the 64-step checkpoints
        W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_cache=True)
    s16 = W.forward_raw(w, q, k, v, a, b, bounded_decay=True)[1]
    with pytest.raises(ValueError):
        W.backward_raw(w, q, k, v, a, b, dy, s16, sa, bounded_decay=True, cache=cache)
