"""GPU dev harness for the WKV7 kernels: parity vs the fp64 oracle and vs the reference kernel
(oracle/_ref), timing of every variant, optional golden-vector minting into gpurun_out/golden.
Run on the GPU box:  python scripts/dev_wkv7.py [--golden] [--time]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import wkv7 as O  # noqa: E402
from oracle import ref_kernel as RK  # noqa: E402
from visualrwkv_b200 import wkv7 as W  # noqa: E402
from visualrwkv_b200 import _lib  # noqa: E402


def run_ours(inp):
    w, q, k, v, a, b, dy = inp
    B, T, H, C = w.shape
    y = torch.empty_like(v)
    s = torch.empty(B, H, T // 16, C, C, dtype=torch.float32, device=w.device)
    sa = torch.empty(B, T, H, C, dtype=torch.float32, device=w.device)
    torch.ops.wind_backstepping.forward(w, q, k, v, a, b, y, s, sa)
    g = [torch.empty_like(w) for _ in range(6)]
    torch.ops.wind_backstepping.backward(w, q, k, v, a, b, dy, s, sa, *g)
    return y, s, sa, g


def parity(shape, kind, seed, fv, bv):
    B, T, H = shape
    cpu = O.make_inputs(B, T, H, 64, seed=seed, kind=kind)
    inp = [x.cuda() for x in cpu]
    W.set_variant(fv, bv)
    y, s, sa, g = run_ours(inp)
    torch.cuda.synchronize()
    y64, s64, sa64 = O.forward(*cpu[:6])
    g64 = O.backward(*cpu, s64, sa64)
    res = {"shape": shape, "kind": kind, "fv": fv, "bv": bv}
    res["y"] = O.err_ratio(y.float().cpu().numpy(), y64)
    res["s"] = O.err_ratio(s.cpu().numpy(), s64)
    res["sa"] = O.err_ratio(sa.cpu().numpy(), sa64)
    res["s_maxrel"] = float(np.max(np.abs(s.cpu().numpy() - s64) / (np.abs(s64) * 1e-3 + 1e-5)))
    res["sa_maxrel"] = float(np.max(np.abs(sa.cpu().numpy() - sa64) / (np.abs(sa64) * 1e-3 + 1e-5)))
    for n, x, r in zip(["dw", "dq", "dk", "dv", "da", "db"], g, g64):
        res[n] = O.err_ratio(x.float().cpu().numpy(), r)
    if RK.available():
        ry, rs, rsa = RK.forward(*inp[:6])
        rg = RK.backward(*inp, rs, rsa)
        torch.cuda.synchronize()
        res["ref_y"] = O.err_ratio(ry.float().cpu().numpy(), y64)
        res["ref_s"] = O.err_ratio(rs.cpu().numpy(), s64)
        for n, x, r in zip(["dw", "dq", "dk", "dv", "da", "db"], rg, g64):
            res["ref_" + n] = O.err_ratio(x.float().cpu().numpy(), r)
        res["y_vs_ref_maxulp"] = int(O.bf16_ulp_diff(y.float().cpu().numpy(), ry.float().cpu().numpy()).max())
        res["y_vs_ref_mismatch"] = float((y != ry).float().mean())
        res["s_vs_ref"] = O.err_ratio(s.cpu().numpy(), rs.cpu().numpy())
        res["sa_vs_ref"] = O.err_ratio(sa.cpu().numpy(), rsa.cpu().numpy())
    return res


from visualrwkv_b200.benchutil import ClockSampler, time_cuda  # noqa: E402


def timeit(fn, iters=30, warm=10):
    med, mn, _ = time_cuda(fn, iters=iters, warmup=warm)
    return float(med), float(mn)


def timing(shape, fvs, bvs):
    B, T, H = shape
    inp = [x.cuda() for x in O.make_inputs(B, T, H, 64, seed=42)]
    w, q, k, v, a, b, dy = inp
    C = 64
    y = torch.empty_like(v)
    s = torch.empty(B, H, T // 16, C, C, dtype=torch.float32, device="cuda")
    sa = torch.empty(B, T, H, C, dtype=torch.float32, device="cuda")
    g = [torch.empty_like(w) for _ in range(6)]
    nel = B * T * H * 64
    out = {"shape": shape}
    for fv in fvs:
        W.set_variant(fv, 1)
        med, mn = timeit(lambda: torch.ops.wind_backstepping.forward(w, q, k, v, a, b, y, s, sa))
        out[f"fwd_v{fv}_ms"] = med
        out[f"fwd_v{fv}_GBs"] = 14 * nel / med / 1e6
    for bv in bvs:
        W.set_variant(1, bv)
        torch.ops.wind_backstepping.forward(w, q, k, v, a, b, y, s, sa)
        med, mn = timeit(lambda: torch.ops.wind_backstepping.backward(w, q, k, v, a, b, dy, s, sa, *g))
        out[f"bwd_v{bv}_ms"] = med
        out[f"bwd_v{bv}_GBs"] = 26 * nel / med / 1e6
    if RK.available():
        med, mn = timeit(lambda: RK.forward(w, q, k, v, a, b), iters=5, warm=2)
        out["ref_fwd_ms"] = med
        ry, rs, rsa = RK.forward(w, q, k, v, a, b)
        med, mn = timeit(lambda: RK.backward(w, q, k, v, a, b, dy, rs, rsa), iters=5, warm=2)
        out["ref_bwd_ms"] = med
    return out


REF_SLICE_SAMPLE = 8192


def mint_golden(outdir):
    """Reference-kernel outputs for fixed seeds (the goldens tests/golden/ is built from)."""
    os.makedirs(outdir, exist_ok=True)
    for name, (B, T, H), kind, seed in [("small_realistic", (2, 64, 3), "realistic", 7),
                                        ("small_stress", (1, 48, 2), "stress", 11)]:
        cpu = O.make_inputs(B, T, H, 64, seed=seed, kind=kind)
        inp = [x.cuda() for x in cpu]
        ry, rs, rsa = RK.forward(*inp[:6])
        rg = RK.backward(*inp, rs, rsa)
        torch.cuda.synchronize()
        d = {"y": ry, "sa": rsa, "s_last": rs[:, :, -1].contiguous()}
        for n, x in zip(["dw", "dq", "dk", "dv", "da", "db"], rg):
            d[n] = x
        arrs = {k2: (v2.view(torch.int16).cpu().numpy() if v2.dtype == torch.bfloat16 else v2.cpu().numpy())
                for k2, v2 in d.items()}
        np.savez_compressed(os.path.join(outdir, f"wkv7_ref_{name}.npz"), B=B, T=T, H=H, seed=seed,
                            kind=np.array(kind), **arrs)
        print("minted", name, {k2: v2.shape for k2, v2 in arrs.items()})

    # the reference kernel's RMS error against the fp64 oracle, which our kernels must not exceed (full tensors)
    B, T, H, seed = 2, 512, 4, 3
    cpu = O.make_inputs(B, T, H, 64, seed=seed)
    inp = [x.cuda() for x in cpu]
    ry, rs, rsa = RK.forward(*inp[:6])
    rg = RK.backward(*inp, rs, rsa)
    torch.cuda.synchronize()
    y64, s64, sa64 = O.forward(*cpu[:6])
    g64 = O.backward(*cpu, s64, sa64)
    errs = {"y": O.err_ratio(ry.float().cpu().numpy(), y64), "s": O.err_ratio(rs.cpu().numpy(), s64)}
    for n, x, r in zip(["dw", "dq", "dk", "dv", "da", "db"], rg, g64):
        errs[n] = O.err_ratio(x.float().cpu().numpy(), r)
    np.savez(os.path.join(outdir, "wkv7_refkernel_errors_b2t512h4.npz"), B=B, T=T, H=H, seed=seed,
             kind=np.array("realistic"), **errs)
    print("minted reference errors", errs)

    # the reference kernel on one (b, h) slice of the cfg2-size inputs, at a fixed sample of REF_SLICE_SAMPLE positions
    # (every output of the slice has 2048 * 64 elements; the checkpoints kept are the chunk-end ones, rs[:, :, 3::4])
    B, T, H, seed, bi, hi = 8, 2048, 12, 42, 3, 5
    sub = [x[bi:bi + 1, :, hi:hi + 1].contiguous().cuda() for x in O.make_inputs(B, T, H, 64, seed=seed)]
    ry, rs, rsa = RK.forward(*sub[:6])
    rg = RK.backward(*sub, rs, rsa)
    torch.cuda.synchronize()
    idx = np.sort(np.random.default_rng(0).choice(T * 64, REF_SLICE_SAMPLE, replace=False)).astype(np.int32)
    d = {"y": ry, "sa": rsa, "s": rs[:, :, 3::4].contiguous()}
    for n, x in zip(["dw", "dq", "dk", "dv", "da", "db"], rg):
        d[n] = x
    arrs = {k2: (v2.view(torch.int16) if v2.dtype == torch.bfloat16 else v2).reshape(-1).cpu().numpy()[idx] for k2, v2 in d.items()}
    rms = {"rms_" + n: float(torch.sqrt(torch.mean(x.double() ** 2))) for n, x in zip(["dw", "dq", "dk", "dv", "da", "db"], rg)}
    np.savez_compressed(os.path.join(outdir, "wkv7_refkernel_slice_b8t2048h12.npz"), B=B, T=T, H=H, seed=seed, b=bi, h=hi,
                        idx=idx, **arrs, **rms)
    print("minted reference slice", {k2: v2.shape for k2, v2 in arrs.items()}, rms)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--golden", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--notest", action="store_true")
    ap.add_argument("--fv", default="1,2")
    ap.add_argument("--bv", default="1,2")
    args = ap.parse_args()
    _lib.load_torch_ops()
    fvs = [int(x) for x in args.fv.split(",")]
    bvs = [int(x) for x in args.bv.split(",")]
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    results = []
    for fv in ([] if args.notest else fvs):
        r = parity((2, 64, 3), "realistic", 7, fv, bvs[min(len(bvs) - 1, fvs.index(fv))])
        print(json.dumps(r)); results.append(r)
    for bv in ([] if args.notest else bvs):
        r = parity((1, 48, 2), "stress", 11, fvs[0], bv)
        print(json.dumps(r)); results.append(r)
    if not args.notest:
        r = parity((2, 512, 4), "realistic", 3, fvs[0], bvs[0])
        print(json.dumps(r)); results.append(r)
    if args.golden and RK.available():
        mint_golden(os.path.join(ROOT, "gpurun_out", "golden"))
    if args.time:
        for shape in [(8, 2048, 12), (4, 2048, 32)]:
            with ClockSampler() as cs:
                r = timing(shape, fvs, bvs)
            r["clocks"] = cs.summary()
            print(json.dumps(r)); results.append(r)
    with open(os.path.join(ROOT, "gpurun_out", "dev_wkv7.json"), "w") as f:
        json.dump(results, f, indent=1)
