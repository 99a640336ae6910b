"""Python front-end of the fused row-wise kernels (csrc/fused_ln.cu, csrc/fused_tmix.cu) and the two
hand-written autograd nodes that orchestrate one RWKV-7 block:

  TmixBlockFn :  x -> x + att(ln1(x))      (VisualRWKV-v7/v7.00/src/model.py:250-251 with :163-195 inside)
  CmixBlockFn :  x -> x + ffn(ln2(x))      (model.py:252 with :221-227 inside)

GEMMs are plain library GEMMs (cuBLAS through torch.matmul / addmm); everything else on the path is one of
our sm_100a kernels reached through the C ABI.  The backward passes are written out by hand (no autograd
tracing inside the block): they call the backward kernels, accumulate residual gradients in the LayerNorm
backward and reduce per-channel parameter gradients from per-CTA fp32 partials.
"""
from __future__ import annotations

import ctypes
import os

import torch
import torch.nn.functional as F

from . import _lib
from . import wkv7 as _wkv7

_c_int, _c_float, _c_void_p, _c_size_t = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


def _p(t):
    return _c_void_p(0 if t is None else t.data_ptr())


def _parr(ts):
    return (_c_void_p * max(len(ts), 1))(*[t.data_ptr() for t in ts])


def _chk(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc}): {_lib.lib().vrwkv_last_error().decode()}")


def _bf16c(*ts):
    for t in ts:
        assert t is None or (t.dtype == torch.bfloat16 and t.is_contiguous() and t.is_cuda), "expected contiguous CUDA bf16"


# ------------------------------------------------------------------------------------------------------
# thin kernel wrappers
# ------------------------------------------------------------------------------------------------------
def _reduce_partials(partial):
    """[blocks, n, C] fp32 -> [n, C] bf16 in one launch (sum over blocks + cast)."""
    L = _lib.lib()
    nb, n, C = partial.shape
    out = torch.empty(n, C, dtype=torch.bfloat16, device=partial.device)
    _chk(L.vrwkv_reduce_partials(_c_int(nb), _c_int(n * C), _p(partial), _p(out), _lib.cur_stream()), "vrwkv_reduce_partials")
    return out


def ln_mix_forward(x2d, T, gamma, beta, eps, coefs, want_h=False):
    """x2d [rows,C] bf16 -> (list of mixed streams, h or None, stats[rows,2] f32)."""
    L = _lib.lib()
    rows, C = x2d.shape
    _bf16c(x2d, gamma, beta, *coefs)
    outs = [torch.empty_like(x2d) for _ in coefs]
    h = torch.empty_like(x2d) if (want_h or not coefs) else None
    stats = torch.empty(rows, 2, dtype=torch.float32, device=x2d.device)
    rc = L.vrwkv_ln_mix_forward(_c_int(rows), _c_int(T), _c_int(C), _c_int(len(coefs)), _c_float(eps), _p(x2d), _p(gamma),
                                _p(beta), _parr(coefs), _parr(outs), _p(h), _p(stats), _lib.cur_stream())
    _chk(rc, "vrwkv_ln_mix_forward")
    return outs, h, stats


def ln_mix_backward(x2d, T, stats, gamma, beta, coefs, douts, dh=None, dresid=None):
    """-> (dx, dgamma, dbeta, [dcoef...]) ; parameter gradients already reduced to bf16."""
    L = _lib.lib()
    rows, C = x2d.shape
    _bf16c(x2d, gamma, beta, dh, dresid, *coefs, *douts)
    nb = L.vrwkv_ln_mix_blocks2(_c_int(rows), _c_int(C))
    partial = torch.empty(nb, 2 + len(coefs), C, dtype=torch.float32, device=x2d.device)
    dx = torch.empty_like(x2d)
    rc = L.vrwkv_ln_mix_backward(_c_int(rows), _c_int(T), _c_int(C), _c_int(len(coefs)), _p(x2d), _p(stats), _p(gamma), _p(beta),
                                 _parr(coefs), _parr(douts), _p(dh), _p(dresid), _p(dx), _p(partial), _lib.cur_stream())
    _chk(rc, "vrwkv_ln_mix_backward")
    red = _reduce_partials(partial)
    return dx, red[0], red[1], [red[2 + i] for i in range(len(coefs))]


def tmix_mid_forward(k, v, vfirst, ww, aa, vv, w0, a0, v0, k_k, k_a):
    L = _lib.lib()
    rows, C = k.shape
    _bf16c(k, v, vfirst, ww, aa, vv, w0, a0, v0, k_k, k_a)
    outs = [torch.empty_like(k) for _ in range(5)]
    rc = L.vrwkv_tmix_mid_forward(_c_int(rows), _c_int(C), _p(k), _p(v), _p(vfirst), _p(ww), _p(aa), _p(vv), _p(w0), _p(a0),
                                  _p(v0), _p(k_k), _p(k_a), *[_p(o) for o in outs], _lib.cur_stream())
    _chk(rc, "vrwkv_tmix_mid_forward")
    return outs  # w, k2, v2, nkk, kka


def tmix_mid_backward(k, v, vfirst, ww, aa, vv, w0, a0, v0, k_k, k_a, dw, dk2, dv2, dnkk, dkka, dk2b=None, dv2b=None):
    L = _lib.lib()
    rows, C = k.shape
    _bf16c(k, v, vfirst, ww, aa, vv, dw, dk2, dv2, dnkk, dkka, dk2b, dv2b)
    has = vfirst is not None
    dk, dv, dww, daa = [torch.empty_like(k) for _ in range(4)]
    dvf = torch.empty_like(k) if has else None
    dvv = torch.empty_like(k) if has else None
    nb = L.vrwkv_tmix_blocks(_c_int(rows))
    partial = torch.empty(nb, 5, C, dtype=torch.float32, device=k.device)
    rc = L.vrwkv_tmix_mid_backward(_c_int(rows), _c_int(C), _p(k), _p(v), _p(vfirst), _p(ww), _p(aa), _p(vv), _p(w0), _p(a0),
                                   _p(v0), _p(k_k), _p(k_a), _p(dw), _p(dk2), _p(dv2), _p(dnkk), _p(dkka), _p(dk2b), _p(dv2b), _p(dk), _p(dv),
                                   _p(dvf), _p(dww), _p(daa), _p(dvv), _p(partial), _lib.cur_stream())
    _chk(rc, "vrwkv_tmix_mid_backward")
    red = _reduce_partials(partial)
    return dk, dv, dvf, dww, daa, dvv, red  # red rows: dw0, da0, dv0, dk_k, dk_a


def tmix_post_forward(y, r, k2, v2, g, gamma, beta, r_k, eps):
    L = _lib.lib()
    rows, C = y.shape
    _bf16c(y, r, k2, v2, g, gamma, beta, r_k)
    z = torch.empty_like(y)
    rc = L.vrwkv_tmix_post_forward(_c_int(rows), _c_int(C), _c_float(eps), _p(y), _p(r), _p(k2), _p(v2), _p(g), _p(gamma),
                                   _p(beta), _p(r_k), _p(z), _lib.cur_stream())
    _chk(rc, "vrwkv_tmix_post_forward")
    return z


def tmix_post_backward(y, r, k2, v2, g, gamma, beta, r_k, eps, dz):
    L = _lib.lib()
    rows, C = y.shape
    _bf16c(y, r, k2, v2, g, dz)
    dy, dr, dk2, dv2, dg = [torch.empty_like(y) for _ in range(5)]
    nb = L.vrwkv_tmix_blocks(_c_int(rows))
    partial = torch.empty(nb, 3, C, dtype=torch.float32, device=y.device)
    rc = L.vrwkv_tmix_post_backward(_c_int(rows), _c_int(C), _c_float(eps), _p(y), _p(r), _p(k2), _p(v2), _p(g), _p(gamma),
                                    _p(beta), _p(r_k), _p(dz), _p(dy), _p(dr), _p(dk2), _p(dv2), _p(dg), _p(partial),
                                    _lib.cur_stream())
    _chk(rc, "vrwkv_tmix_post_backward")
    red = _reduce_partials(partial)
    return dy, dr, dk2, dv2, dg, red  # red rows: dgamma, dbeta, dr_k


def relu_sq_forward(x):
    L = _lib.lib()
    _bf16c(x)
    y = torch.empty_like(x)
    _chk(L.vrwkv_relu_sq_forward(_c_size_t(x.numel()), _p(x), _p(y), _lib.cur_stream()), "vrwkv_relu_sq_forward")
    return y


def relu_sq_backward(x, dy):
    L = _lib.lib()
    _bf16c(x, dy)
    dx = torch.empty_like(x)
    _chk(L.vrwkv_relu_sq_backward(_c_size_t(x.numel()), _p(x), _p(dy), _p(dx), _lib.cur_stream()), "vrwkv_relu_sq_backward")
    return dx


def relu_sq_backward_from_act(act, dy):
    L = _lib.lib()
    _bf16c(act, dy)
    dx = torch.empty_like(act)
    _chk(L.vrwkv_relu_sq_backward_from_act(_c_size_t(act.numel()), _p(act), _p(dy), _p(dx), _lib.cur_stream()),
         "vrwkv_relu_sq_backward_from_act")
    return dx


# Which WKV7 kernels the fused time-mix block runs (bench.py --wkv, env VRWKV_WKV_PATH).  The block builds
# w = -softplus(.) - 0.5 itself (tmix_mid_fwd_kernel, model.py:176), so it may promise bounded decay.
#   "x6"   : chunk-parallel tensor-core forward with bf16-split products (wkv7_x6_fwd.cuh) + the matching backward —
#            fp32-level accuracy, passes the same element-wise parity asserts as the step-by-step kernels (default);
#   "step" : the step-by-step fp32 kernels (wkv7_fwd2/bwd2.cuh), what torch.ops.wind_backstepping binds;
#   "tf32" : the round-1 single-pass TF32 chunk kernels (faster products, sa/s only to ~5e-4: comparison only).
WKV_PATH = os.environ.get("VRWKV_WKV_PATH", "x6")
X3_BACKWARD = True   # the x3 chunked backward reads one checkpoint per 64-step chunk (a quarter of the checkpoint traffic)


def set_wkv_path(path: str) -> None:
    global WKV_PATH
    assert path in ("x6", "step", "tf32"), path
    WKV_PATH = path


def wkv7_fwd_raw(w, q, k, v, a, b):
    """[B,T,H,64] bf16 x6 -> y, s, sa, cache (the x6 path's chunk cache for wkv7_bwd_raw; None on the other paths)."""
    if WKV_PATH == "tf32":
        return (*_wkv7.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True, tf32=True), None)
    if WKV_PATH == "x6":
        if X3_BACKWARD and w.shape[1] % _wkv7.CHUNK == 0:
            # the backward then loads each chunk's masked matrices and inverse instead of recomputing them (other T take
            # the step-by-step kernels, which have no cache)
            return _wkv7.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True, chunk_cache=True)
        return (*_wkv7.forward_raw(w, q, k, v, a, b, bounded_decay=True), None)
    return (*_wkv7.forward_raw(w, q, k, v, a, b), None)


def wkv7_bwd_raw(w, q, k, v, a, b, dy, s, sa, cache=None):
    return _wkv7.backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay=(WKV_PATH != "step"), tf32=(WKV_PATH == "tf32"),
                              cache=cache)


# ------------------------------------------------------------------------------------------------------
# plain LayerNorm node (ln0, ln_out, proj.ln_v)
# ------------------------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps):
        shp = x.shape
        x2 = x.reshape(-1, shp[-1]).contiguous()
        _, h, stats = ln_mix_forward(x2, x2.shape[0], weight, bias, eps, [], want_h=True)
        ctx.save_for_backward(x2, stats, weight, bias)
        ctx.shp = shp
        return h.view(shp)

    @staticmethod
    def backward(ctx, dh):
        x2, stats, weight, bias = ctx.saved_tensors
        dh2 = dh.reshape(x2.shape).contiguous()
        dx, dg, db, _ = ln_mix_backward(x2, x2.shape[0], stats, weight, bias, [], [], dh=dh2)
        return dx.view(ctx.shp), dg, db, None


# ------------------------------------------------------------------------------------------------------
# time-mix half block
# ------------------------------------------------------------------------------------------------------
_TM_PARAMS = ["x_r", "x_w", "x_k", "x_v", "x_a", "x_g", "w0", "w1", "w2", "a0", "a1", "a2", "v0", "v1", "v2", "g1", "g2",
              "k_k", "k_a", "r_k"]


class TmixBlockFn(torch.autograd.Function):
    """(x, v_first, ln1.w, ln1.b, <20 att params>, Wr, Wk, Wv, Wo, lnx.w, lnx.b) -> (x + att(ln1(x)), v_first)."""

    @staticmethod
    def forward(ctx, x, v_first, ln_w, ln_b, x_r, x_w, x_k, x_v, x_a, x_g, w0, w1, w2, a0, a1, a2, v0, v1, v2, g1, g2, k_k, k_a,
                r_k, Wr, Wk, Wv, Wo, lnx_w, lnx_b, layer_id, n_head, ln_eps, gn_eps, with_ln):
        B, T, C = x.shape
        rows = B * T
        x2 = x.reshape(rows, C).contiguous()
        coefs = [c.reshape(C) for c in (x_r, x_w, x_k, x_v, x_a, x_g)]
        (xr, xw, xk, xv, xa, xg), _, stats = ln_mix_forward(x2, T, ln_w if with_ln else None, ln_b if with_ln else None, ln_eps, coefs)
        own = gemm2_supported(rows, C, C)   # CTA-pair tcgen05 GEMMs (csrc/gemm2_sm100.cu); cuBLAS only for shapes it cannot tile
        if own:
            r, k, v = gemm2_grouped([xr, xk, xv], [Wr, Wk, Wv])   # one launch: 3 x (rows x C x C)
        else:
            r = xr @ Wr.t()
            k = xk @ Wk.t()
            v = xv @ Wv.t()
        has_vres = layer_id != 0
        vf2 = v_first.reshape(rows, C).contiguous() if has_vres else None
        lora_own = own and _lora_ok(w1, a1, g1, v1 if has_vres else None)
        if lora_own:
            # the LoRA branches (model.py:176,181-184) as two grouped launches (ranks differ per branch; the launch tiles the
            # widest and TMA zero-fills the rest): down-projections with their activation in the epilogue, then up-projections
            downs = [(xw, w1, ACT_TANH), (xa, a1, ACT_NONE), (xg, g1, ACT_SIGMOID)] + ([(xv, v1, ACT_NONE)] if has_vres else [])
            ups = [w2, a2, g2] + ([v2] if has_vres else [])
            hs = gemm2_grouped([xx for xx, _, _ in downs], [wd for _, wd, _ in downs], G2_NN, EPI_ACT, acts=[ac for _, _, ac in downs])
            outs = gemm2_grouped(hs, ups, G2_NN)
            hw, ha, hg = hs[:3]
            ww, aa, g = outs[:3]
            hv, vv = (hs[3], outs[3]) if has_vres else (None, None)
        else:
            hw = torch.tanh(xw @ w1)
            ww = hw @ w2
            ha = xa @ a1
            aa = ha @ a2
            hg = torch.sigmoid(xg @ g1)
            g = hg @ g2
            if has_vres:
                hv = xv @ v1
                vv = hv @ v2
            else:
                hv = vv = None
        w, k2, v2_, nkk, kka = tmix_mid_forward(k, v, vf2, ww, aa, vv, w0.reshape(C), a0.reshape(C),
                                                v0.reshape(C) if has_vres else None, k_k.reshape(C), k_a.reshape(C))
        H = n_head
        v4 = lambda t: t.view(B, T, H, 64)
        y, s, sa, wcache = wkv7_fwd_raw(v4(w), v4(r), v4(k2), v4(v2_), v4(nkk), v4(kka))
        z = tmix_post_forward(y.view(rows, C), r, k2, v2_, g, lnx_w, lnx_b, r_k.reshape(C), gn_eps)
        if own:
            out = gemm2(z, Wo, G2_TN, EPI_ADD, x2) if with_ln else gemm2(z, Wo)
        else:
            out = torch.addmm(x2, z, Wo.t()) if with_ln else z @ Wo.t()
        ctx.save_for_backward(x2, stats, ln_w, ln_b, *coefs, xr, xw, xk, xv, xa, xg, r, k, v, hw, ww, ha, aa, hg, g, hv, vv, vf2,
                              w, k2, v2_, nkk, kka, y, s, sa, wcache, z, w0, w1, w2, a0, a1, a2, v0, v1, v2, g1, g2, k_k, k_a, r_k,
                              Wr, Wk, Wv, Wo, lnx_w, lnx_b)
        ctx.meta = (B, T, C, H, layer_id, ln_eps, gn_eps, with_ln)
        ctx.lora_own = lora_own
        v_out = v.view(B, T, C)  # layer 0: this is v_first; later layers: ignored by the caller
        if has_vres:
            ctx.mark_non_differentiable(v_out)
        return out.view(B, T, C), v_out

    @staticmethod
    def backward(ctx, dout, dvfirst_out):
        (x2, stats, ln_w, ln_b, c_r, c_w, c_k, c_v, c_a, c_g, xr, xw, xk, xv, xa, xg, r, k, v, hw, ww, ha, aa, hg, g, hv, vv, vf2,
         w, k2, v2_, nkk, kka, y, s, sa, wcache, z, w0, w1, w2, a0, a1, a2, v0, v1, v2, g1, g2, k_k, k_a, r_k, Wr, Wk, Wv, Wo,
         lnx_w, lnx_b) = ctx.saved_tensors
        B, T, C, H, layer_id, ln_eps, gn_eps, with_ln = ctx.meta
        rows = B * T
        has_vres = layer_id != 0
        do = dout.reshape(rows, C).contiguous()
        own = gemm2_supported(rows, C, C) and gemm2_supported(C, C, rows)
        dz = gemm2(do, Wo, G2_NN) if own else do @ Wo
        dy, dr, dk2a, dv2a, dg, red3 = tmix_post_backward(y.view(rows, C), r, k2, v2_, g, lnx_w, lnx_b, r_k.reshape(C), gn_eps, dz)
        v4 = lambda t: t.view(B, T, H, 64)
        dw, dq, dk2b, dv2b, dnkk, dkka = wkv7_bwd_raw(v4(w), v4(r), v4(k2), v4(v2_), v4(nkk), v4(kka), v4(dy), s, sa, wcache)
        dr.add_(dq.view(rows, C))
        dk, dv, dvf, dww, daa, dvv, red5 = tmix_mid_backward(
            k, v, vf2, ww, aa, vv, w0.reshape(C), a0.reshape(C), v0.reshape(C) if has_vres else None, k_k.reshape(C),
            k_a.reshape(C), dw.view(rows, C), dk2a, dv2a, dnkk.view(rows, C), dkka.view(rows, C), dk2b.view(rows, C), dv2b.view(rows, C))
        if not has_vres and dvfirst_out is not None:
            dv.add_(dvfirst_out.reshape(rows, C))
        # LoRA branches
        if ctx.lora_own:
            douts = [dww, daa, dg] + ([dvv] if has_vres else [])
            hs = [hw, ha, hg] + ([hv] if has_vres else [])
            xs = [xw, xa, xg] + ([xv] if has_vres else [])
            downs = [w1, a1, g1] + ([v1] if has_vres else [])
            ups = [w2, a2, g2] + ([v2] if has_vres else [])
            acts = [ACT_TANH, ACT_NONE, ACT_SIGMOID] + ([ACT_NONE] if has_vres else [])
            ng, Rp = len(hs), max(h.shape[1] for h in hs)
            dps = gemm2_grouped(douts, ups, G2_TN, EPI_ACT_BWD, residuals=hs, acts=acts)        # d(pre-activation) [rows, rank]
            dxl = gemm2_grouped(dps, downs, G2_TN)                                              # [rows, C]
            # h^T dout [rank, C], computed as (dout^T h)^T: with the rank as the M extent half of every 256-row pair tile is
            # padding and the launch ran 1.6x (warm) to 3x (cold) slower than its mirror image below (scripts/dev_lora.py)
            dU = gemm2_grouped(douts, hs, G2_TT, ksplit=min(4, _ksplit(ng, C, Rp, rows)), transposed=[1] * ng)
            dD = gemm2_grouped(xs, dps, G2_TT, ksplit=min(4, _ksplit(ng, C, Rp, rows)))         # x^T dpre [C, rank]
            dw2, da2, dg2 = dU[:3]
            dw1, da1, dg1 = dD[:3]
            dxw, dxa, dxg = dxl[:3]
            if has_vres:
                dv2p, dv1, dxv_lora = dU[3], dD[3], dxl[3]
            else:
                dv2p = dv1 = dxv_lora = None
        else:
            dhg = dg @ g2.t()
            dg2 = hg.t() @ dg
            dpg = torch.ops.aten.sigmoid_backward(dhg, hg)
            dxg = dpg @ g1.t()
            dg1 = xg.t() @ dpg
            dhw = dww @ w2.t()
            dw2 = hw.t() @ dww
            dpw = torch.ops.aten.tanh_backward(dhw, hw)
            dxw = dpw @ w1.t()
            dw1 = xw.t() @ dpw
            dha = daa @ a2.t()
            da2 = ha.t() @ daa
            dxa = dha @ a1.t()
            da1 = xa.t() @ dha
            if has_vres:
                dhv = dvv @ v2.t()
                dv2p = hv.t() @ dvv
                dv1 = xv.t() @ dhv
                dxv_lora = dhv @ v1.t()
            else:
                dv2p = dv1 = dxv_lora = None
        # main projections
        if own:
            # dgrad: dx = dy W (W is [out, in]: contraction over its rows); wgrad: dW = dy^T x over the token rows, the
            # four C x C weight gradients of the block in one split-K launch
            if has_vres:
                dxr, dxk = gemm2_grouped([dr, dk], [Wr, Wk], G2_NN)
                dxv = gemm2(dv, Wv, G2_NN, EPI_ADD, dxv_lora)
            else:
                dxr, dxk, dxv = gemm2_grouped([dr, dk, dv], [Wr, Wk, Wv], G2_NN)
            dWo, dWr, dWk, dWv = gemm2_grouped([do, dr, dk, dv], [z, xr, xk, xv], G2_TT, ksplit=_ksplit(4, C, C, rows))
        else:
            dWo = do.t() @ z
            dxr = dr @ Wr
            dWr = dr.t() @ xr
            dxk = dk @ Wk
            dWk = dk.t() @ xk
            dWv = dv.t() @ xv
            dxv = torch.addmm(dxv_lora, dv, Wv) if has_vres else dv @ Wv
        coefs = [c_r, c_w, c_k, c_v, c_a, c_g]
        dx, dlnw, dlnb, dco = ln_mix_backward(x2, T, stats, ln_w if with_ln else None, ln_b if with_ln else None, coefs,
                                              [dxr, dxw, dxk, dxv, dxa, dxg], dresid=do if with_ln else None)
        sh = lambda t: t.view(1, 1, C)
        grads = [dx.view(B, T, C), dvf.view(B, T, C) if has_vres else None,
                 dlnw if with_ln else None, dlnb if with_ln else None,
                 sh(dco[0]), sh(dco[1]), sh(dco[2]), sh(dco[3]), sh(dco[4]), sh(dco[5]),
                 sh(red5[0]), dw1, dw2, sh(red5[1]), da1, da2,
                 sh(red5[2]) if has_vres else None, dv1, dv2p, dg1, dg2, sh(red5[3]), sh(red5[4]),
                 red3[2].view(H, 64), dWr, dWk, dWv, dWo, red3[0], red3[1],
                 None, None, None, None, None]
        return tuple(grads)


class CmixBlockFn(torch.autograd.Function):
    """(x, ln2.w, ln2.b, x_k, Wkey, Wval) -> x + value(relu(key(mix(ln2(x))))^2)."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, x_k, Wkey, Wval, ln_eps, with_ln):
        B, T, C = x.shape
        rows = B * T
        x2 = x.reshape(rows, C).contiguous()
        ck = x_k.reshape(C)
        (xk,), _, stats = ln_mix_forward(x2, T, ln_w if with_ln else None, ln_b if with_ln else None, ln_eps, [ck])
        M, Hd = rows, Wkey.shape[0]
        if gemm2_supported(M, Hd, C) and gemm2_supported(M, C, Hd):
            # key GEMM with relu^2 in the tcgen05 epilogue (the 4C-wide pre-activation never touches HBM), value GEMM
            # with the residual add in the epilogue
            act = gemm2(xk, Wkey, G2_TN, EPI_RELU_SQ)
            out = gemm2(act, Wval, G2_TN, EPI_ADD, x2) if with_ln else gemm2(act, Wval)
            hk = None
        else:
            hk = xk @ Wkey.t()
            act = relu_sq_forward(hk)
            out = torch.addmm(x2, act, Wval.t()) if with_ln else act @ Wval.t()
        ctx.save_for_backward(x2, stats, ln_w, ln_b, ck, xk, hk, act, Wkey, Wval)
        ctx.meta = (B, T, C, with_ln)
        return out.view(B, T, C)

    @staticmethod
    def backward(ctx, dout):
        x2, stats, ln_w, ln_b, ck, xk, hk, act, Wkey, Wval = ctx.saved_tensors
        B, T, C, with_ln = ctx.meta
        do = dout.reshape(B * T, C).contiguous()
        rows, Hd = B * T, Wkey.shape[0]
        if hk is None and gemm2_supported(rows, Hd, C) and gemm2_supported(rows, C, Hd) and gemm2_supported(C, Hd, rows) and gemm2_supported(Hd, C, rows):
            dhk = gemm2(do, Wval, G2_NN, EPI_RELUSQ_BWD, act)     # dact = do Wval and d relu()^2 in one pass: dact never reaches HBM
            dxk = gemm2(dhk, Wkey, G2_NN)
            # both weight gradients in one launch of C x 4C problems: dWval = do^T act, dWkey = (xk^T dhk)^T (stored transposed)
            dWval, dWkey = gemm2_grouped([do, xk], [act, dhk], G2_TT, ksplit=1, transposed=[0, 1])
        else:
            dact = do @ Wval
            dWval = do.t() @ act
            dhk = relu_sq_backward(hk, dact) if hk is not None else relu_sq_backward_from_act(act, dact)
            dxk = dhk @ Wkey
            dWkey = dhk.t() @ xk
        dx, dlnw, dlnb, dco = ln_mix_backward(x2, T, stats, ln_w if with_ln else None, ln_b if with_ln else None, [ck], [dxk],
                                              dresid=do if with_ln else None)
        return (dx.view(B, T, C), dlnw if with_ln else None, dlnb if with_ln else None, dco[0].view(1, 1, C),
                dWkey, dWval, None, None)


# ------------------------------------------------------------------------------------------------------
# head + shifted cross-entropy + L2Wrap  (model.py:323-325, :418-434, :257-271)
# ------------------------------------------------------------------------------------------------------
class HeadLossFn(torch.autograd.Function):
    """(features [B,T,C] after ln_out, head weight [V,C], labels [B,T]) -> scalar training loss.

    logits = x W^T is one CTA-pair tcgen05 GEMM (gemm2); the shifted CE (per-sample mean over valid labels, mean over the batch) and
    the L2Wrap term are evaluated in ONE pass over the logits, and the backward overwrites the logits buffer with
    d(loss)/d(logits) in one more pass — instead of the ~10 passes over the 2.1 GB tensor the eager graph makes."""

    @staticmethod
    def forward(ctx, x, weight, labels, ignore_index):
        L = _lib.lib()
        B, T, C = x.shape
        V = weight.shape[0]
        rows = B * T
        x2 = x.reshape(rows, C).contiguous()
        own = HEAD_OWN_GEMM and gemm2_supported(rows, V, C) and gemm2_supported(V, C, rows) and gemm2_supported(rows, C, V)
        logits = gemm2(x2, weight) if own else x2 @ weight.t()
        labels = labels.contiguous()
        assert labels.dtype == torch.int64 and labels.shape == (B, T)
        lse = torch.empty(rows, dtype=torch.float32, device=x.device)
        rmax = torch.empty_like(lse)
        nll = torch.empty_like(lse)
        amax = torch.empty(rows, dtype=torch.int32, device=x.device)
        _chk(L.vrwkv_ce_forward(_c_int(rows), _c_int(T), _c_int(V), _c_int(ignore_index), _p(logits), _p(labels), _p(lse), _p(rmax),
                                _p(amax), _p(nll), _lib.cur_stream()), "vrwkv_ce_forward")
        valid = (labels[:, 1:] != ignore_index).sum(1).clamp(min=1).float()          # [B]
        loss = (nll.view(B, T).sum(1) / valid).mean()
        ctx.save_for_backward(x2, weight, logits, labels, lse, rmax, amax, valid)
        ctx.meta = (B, T, C, V, ignore_index)
        ctx.logits_consumed = False
        return loss.to(x.dtype)   # the reference's F.cross_entropy on bf16 logits returns a bf16 loss too (model.py:430-434)

    @staticmethod
    def backward(ctx, gloss):
        L = _lib.lib()
        x2, weight, logits, labels, lse, rmax, amax, valid = ctx.saved_tensors
        B, T, C, V, ignore_index = ctx.meta
        rows = B * T
        if ctx.logits_consumed:
            # the first backward turned the saved logits into d(loss)/d(logits) in place (one buffer of B*T*V bf16 instead of
            # two); a second pass over the same graph (retain_graph=True) would read gradients as logits
            raise RuntimeError("HeadLossFn: backward called twice on the same forward (the logits buffer was reused for the "
                               "gradient); run the forward again instead of retain_graph=True")
        ctx.logits_consumed = True
        has_t = torch.ones(B, T, dtype=torch.bool, device=x2.device)
        has_t[:, -1] = False
        has_t[:, :-1] &= labels[:, 1:] != ignore_index
        wrow = (has_t.float() * (gloss.float() / (valid * B)).view(B, 1)).reshape(rows).contiguous()
        l2 = 1e-4 / (B * T)
        _chk(L.vrwkv_ce_backward(_c_int(rows), _c_int(T), _c_int(V), _c_int(ignore_index), _p(logits), _p(labels), _p(lse), _p(rmax),
                                 _p(amax), _p(wrow), _c_float(l2), _lib.cur_stream()), "vrwkv_ce_backward")
        dlogits = logits  # overwritten in place
        if HEAD_OWN_GEMM and gemm2_supported(rows, V, C) and gemm2_supported(V, C, rows) and gemm2_supported(rows, C, V):
            dx = gemm2(dlogits, weight, G2_NN)
            dW = gemm2(dlogits, x2, G2_TT, ksplit=_ksplit(1, V, C, rows))
        else:
            dx = dlogits @ weight
            dW = dlogits.t() @ x2
        return dx.view(B, T, C), dW, None, None


# ------------------------------------------------------------------------------------------------------
# tcgen05 GEMM with fused epilogues (csrc/gemm_sm100.cu)
# ------------------------------------------------------------------------------------------------------
EPI_NONE, EPI_RELU_SQ, EPI_ADD = 0, 1, 2


def gemm_tn(a, w, epilogue=EPI_NONE, residual=None):
    """C[M,N] = epilogue(a[M,K] @ w[N,K]^T) on the tcgen05 tensor cores (bf16 in, fp32 accumulate, bf16 out)."""
    L = _lib.lib()
    _bf16c(a, w, residual)
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K
    c = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    _chk(L.vrwkv_gemm_bf16_tn(_c_int(M), _c_int(N), _c_int(K), _p(a), _p(w), _p(c), _c_int(epilogue), _p(residual),
                              _lib.cur_stream()), "vrwkv_gemm_bf16_tn")
    return c


def gemm_supported(M, N, K):
    return K % 64 == 0 and N % 128 == 0 and M > 0


# ------------------------------------------------------------------------------------------------------
# CTA-pair tcgen05 GEMM, all layouts (csrc/gemm2_sm100.cu)
# ------------------------------------------------------------------------------------------------------
G2_TN, G2_NN, G2_TT = 0, 2, 3     # layout bits: 1 = A stored [K,M], 2 = B stored [K,N]


EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_ADD, EPI_ACT, EPI_ACT_BWD = 5, 6, 7, 8, 9
ACT_NONE, ACT_TANH, ACT_SIGMOID = 0, 1, 2


def gemm2_grouped(As, Bs, layout=G2_TN, epilogue=EPI_NONE, residuals=None, ksplit=1, transposed=None, biases=None, r_rows=0, acts=None):
    """[epilogue(op(a) . op(b)) for a, b in zip(As, Bs)] in ONE launch, bf16 in / out, fp32 accumulate.
      G2_TN: a [M,K], b [N,K]  -> a @ b.T      (forward y = x W^T)
      G2_NN: a [M,K], b [K,N]  -> a @ b        (dgrad  dx = dy W)
      G2_TT: a [K,M], b [K,N]  -> a.T @ b      (wgrad  dW = dy^T x; ksplit > 1 slices the long contraction)
    Groups may differ in shape (the LoRA ranks): the launch tiles the largest, rounded up to the tile, and each group's
    tensors keep their own exact size."""
    L = _lib.lib()
    _bf16c(*As, *Bs, *(residuals or []), *(biases or []))
    a_mn, b_mn = layout & 1, (layout >> 1) & 1
    dims = []
    for a, b in zip(As, Bs):
        Mg, Kg = (a.shape[1], a.shape[0]) if a_mn else a.shape
        Ng, Kb = (b.shape[1], b.shape[0]) if b_mn else b.shape
        assert Kb == Kg, (a.shape, b.shape)
        dims.append((Mg, Ng, Kg))
    M = max(d[0] for d in dims)
    N = -(-max(d[1] for d in dims) // 128) * 128
    K = -(-max(d[2] for d in dims) // (64 * ksplit)) * (64 * ksplit)
    ragged = any(d != (M, N, K) for d in dims)
    tr = list(transposed) if transposed else [0] * len(As)
    dev = As[0].device
    Cs = [torch.empty((Ng, Mg) if t else (Mg, Ng), dtype=torch.bfloat16, device=dev) for t, (Mg, Ng, _) in zip(tr, dims)]   # transposed[g]: (a.b)^T
    flat = [v for d in dims for v in d]
    _chk(L.vrwkv_gemm2_bf16_grouped(_c_int(M), _c_int(N), _c_int(K), _c_int(len(As)), _parr(As), _parr(Bs), _parr(Cs),
                                    _parr(residuals) if residuals else None, (_c_int * len(tr))(*tr), _c_int(layout), _c_int(epilogue),
                                    _c_int(ksplit), _parr(biases) if biases else None, _c_int(r_rows),
                                    (_c_int * len(acts))(*acts) if acts else None, (_c_int * len(flat))(*flat) if ragged else None,
                                    _lib.cur_stream()),
         "vrwkv_gemm2_bf16_grouped")
    return Cs

def gemm2(a, b, layout=G2_TN, epilogue=EPI_NONE, residual=None, ksplit=1, bias=None, r_rows=0):
    return gemm2_grouped([a], [b], layout, epilogue, [residual] if residual is not None else None, ksplit,
                         biases=[bias] if bias is not None else None, r_rows=r_rows)[0]


EPI_RELUSQ_BWD = 4
HEAD_OWN_GEMM = os.environ.get("VRWKV_HEAD_GEMM", "own") == "own"   # "cublas": library GEMMs for the three head products


def gemm2_supported(M, N, K, ksplit=1):
    """Extents the CTA-pair GEMM takes: multiples of 8 (16-byte TMA row strides); tiles past the edge are zero-filled / clipped."""
    return K % 8 == 0 and N % 8 == 0 and M % 8 == 0 and M > 0


def _lora_ok(*downs):
    """The LoRA ranks the grouped launches take: multiples of 8 (TMA row strides of 16 bytes)."""
    return all(d.shape[1] % 8 == 0 for d in downs if d is not None)


def _ksplit(groups, M, N, K):
    """Slices of the contraction for a weight gradient: enough (group, tile, slice) items for the 74 CTA pairs.  When
    halving the tile width (the C library does that by itself for an unsplit weight gradient with fewer than 60 tiles)
    already fills the machine, no split: the fp32-atomic meeting of slices costs a fixed ~35 us per launch."""
    tiles = groups * ((M + 255) // 256) * (N // (256 if N % 256 == 0 else 128))
    if N % 256 == 0 and tiles < 60 and 2 * tiles >= 60:
        return 1
    ks = 1
    while ks < 8 and tiles * ks < 74 and K % (64 * ks * 2) == 0:
        ks *= 2
    return ks


# ------------------------------------------------------------------------------------------------------
# image -> language projector  (MLPWithContextGating, model.py:328-338; the LayerNorm after it is LayerNormFn)
# ------------------------------------------------------------------------------------------------------
class ProjectorFn(torch.autograd.Function):
    """(x [rows, Dv], gate.weight [Dv, Dv], o_proj.weight [C, Dv]) -> o_proj(x * sigmoid(gate(x))) [rows, C]."""

    @staticmethod
    def forward(ctx, x, Wg, Wo):
        L = _lib.lib()
        g = gemm2(x, Wg)
        h = torch.empty_like(x)
        _chk(L.vrwkv_sigmul_forward(_c_size_t(x.numel()), _p(x), _p(g), _p(h), _lib.cur_stream()), "vrwkv_sigmul_forward")
        o = gemm2(h, Wo)
        ctx.save_for_backward(x, g, h, Wg, Wo)
        return o

    @staticmethod
    def backward(ctx, do):
        L = _lib.lib()
        x, g, h, Wg, Wo = ctx.saved_tensors
        rows, Dv = x.shape
        C = Wo.shape[0]
        do = do.contiguous()
        dh = gemm2(do, Wo, G2_NN)
        dWo = gemm2(do, h, G2_TT, ksplit=_ksplit(1, C, Dv, rows))
        need_dx = ctx.needs_input_grad[0]
        dx1 = torch.empty_like(x) if need_dx else None
        dg = torch.empty_like(x)
        _chk(L.vrwkv_sigmul_backward(_c_size_t(x.numel()), _p(x), _p(g), _p(dh), _p(dx1), _p(dg), _lib.cur_stream()), "vrwkv_sigmul_backward")
        dWg = gemm2(dg, x, G2_TT, ksplit=_ksplit(1, Dv, Dv, rows))
        dx = gemm2(dg, Wg, G2_NN, EPI_ADD, dx1) if need_dx else None
        return dx, dWg, dWo
