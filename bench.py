#!/usr/bin/env python
"""bench.py — the reference's headline metric on its own config, measured on B200.

metric : tokens/s, fwd+bwd (+ grad all-reduce + optimizer step), whole job over N GPUs
workload (N=1, BASELINE.json configs[1]): RWKV-x070 0.1B (L12 C768 H12) + SigLIP-B/16 @224 -> 196 patches
         -> AdaptiveAvgPool to 576 image tokens, ctx 2048, batch 8 per GPU, bf16, synthetic data,
         reference init (zero-init tensors re-randomised, SURVEY.md §8d).
Multi-GPU: pure data parallelism, one process per GPU (torchrun), weak scaling (batch 8 per GPU), one
         bucketed bf16 gradient all-reduce per step over NCCL.

One JSON line on rank 0 (see the task contract): value (inputs resident in HBM), e2e (pinned-host
inputs copied H2D and the loss read back D2H inside the timed region, through the public
VisualRWKV.training_step API), roofline of the dominant hand-written kernel (WKV7 backward; the forward
is reported next to it) timed live with CUDA events on the launching stream, cpu_baseline (the oracle
port on the host cores, bounded sample), clocks.

`--impl reference` times the reference's own CPU implementation of the path — the oracle port, since
the reference has no CPU path for x070 (SURVEY.md §0.1) and its model.py cannot be imported without
CUDA/Lightning/DeepSpeed/timm — on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WKV_FWD_BYTES_PER_ELEM = 14  # 6 bf16 reads + 1 bf16 write (BASELINE.md §2.4)
WKV_BWD_BYTES_PER_ELEM = 26  # 7 bf16 reads + 6 bf16 writes
# The WKV7 kernels behind each --wkv path, and dram__bytes_read.sum + dram__bytes_write.sum per launch at cfg2
# (B8 T2048 C768) from the ncu --set full captures named beside them (profiles/); None = not captured for this build.
WKV_PATHS = {
    "x6": {"fwd": "wkv7_x6_fwd_kernel<chunk checkpoints>", "bwd": "wkv7_x3_bwd_kernel",
           "traffic_fwd": int((151.093 + 84.057) * 1e6), "traffic_bwd": int((275.737 + 126.352) * 1e6), "ncu": "profiles/r2_ncu_summary.csv"},
    "step": {"fwd": "wkv7_fwd2_kernel<4,4>", "bwd": "wkv7_bwd2_kernel<4,3>", "traffic_fwd": int((151 + 226) * 1e6), "traffic_bwd": None,
             "ncu": "profiles/r1b_*"},
    "tf32": {"fwd": "wkv7_chunk_fwd_kernel<chunk checkpoints>", "bwd": "wkv7_chunk_dstate_kernel + wkv7_chunk_bwd_kernel",
             "traffic_fwd": int((151.359 + 83.432) * 1e6), "traffic_bwd": int((121.974 + 22.821 + 324.469 + 168.727) * 1e6),
             "ncu": "profiles/r1e_wkv7_tc_model_path_summary.csv"},
}
CONFIGS = {   # BASELINE.json configs[1] and configs[2] (one GPU's share)
    "cfg2": dict(layers=12, embd=768, batch=8, ctx=2048, name="RWKV-x070 0.1B (L12 C768 H12 N64)"),
    "cfg3": dict(layers=24, embd=2048, batch=4, ctx=2048, name="RWKV-x070 1.5B (L24 C2048 H32 N64)"),
}
LORA_RANKS = {768: 64 + 64 + 32 + 128, 2048: 96 + 96 + 64 + 256}   # v7.00/src/model.py:118,127,133,140 (w, a, v, g)
DUMP_SAMPLE = 16384   # elements written per tensor by --dump-outputs: ~24 MB for the 402 trainable tensors of cfg2


def dump_outputs(out_dir, loss, named_params):
    """What a caller of the timed step holds after its last step: the loss and, for every trainable parameter, its
    gradient and its updated value, each as DIR/<kind>.<parameter name>.npy in float32.  A tensor of more than
    DUMP_SAMPLE elements is reduced to a sample whose positions depend only on the parameter's name and size, so runs
    with the same arguments (and therefore the same seeded inputs) can be compared file by file across builds.  Compare
    with a tolerance: the bf16 gradients are not bitwise reproducible from run to run (at cfg2 on a B200 at 1000 W, two
    runs of the same build differed by a median 0.7 % relative RMS over the gradient files, 1.7 % at most, with equal
    losses)."""
    import zlib

    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    for name, p in named_params:
        idx = None
        if p.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(0, p.numel(), (DUMP_SAMPLE,), generator=g).to(p.device)
        for kind, t in (("grad", p.grad), ("param", p)):
            if t is None:
                continue
            flat = t.detach().reshape(-1)
            if idx is not None:
                flat = flat[idx]
            np.save(os.path.join(out_dir, f"{kind}.{name}.npy"), flat.float().cpu().numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# --------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) — shared by cpu_baseline and --impl reference
# --------------------------------------------------------------------------------------------------
def cpu_reference_run(steps: int, warmup: int, T: int = 512, B: int = 1, n_img_tok: int = 196):
    """fp32 restatement of the same model (0.1B + SigLIP-B/16@224) on the host cores, fwd+bwd, on BASELINE.json
    configs[0]: one 224x224 image (196 patch tokens, identity pooling), ctx 512, batch 1 (SURVEY.md §8d(ii))."""
    from oracle import model_ref as MR
    from visualrwkv_b200.model import VisualRWKV, default_args, randomize_zero_init
    # small-operator workload: beyond ~32 threads the fork/join cost of every op outweighs the parallelism (on the
    # 128-core GPU hosts the 128-thread run was 5x slower than this), so the baseline uses min(cores, 32) threads
    ncores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(ncores)
    os.environ["OMP_NUM_THREADS"] = str(ncores)
    torch.manual_seed(0)
    args = default_args(num_token_per_image=n_img_tok, ctx_len=T)
    model = VisualRWKV(args)
    randomize_zero_init(model)
    P = {}
    for k, v in model.state_dict().items():
        t = v.detach().float().clone()
        if not k.startswith("vit.") and "emb.weight" not in k:
            t.requires_grad_(True)
        P[k] = t
    cfg = {"vit": model.vit.cfg, "num_token_per_image": n_img_tok, "n_layer": args.n_layer, "n_head": args.dim_att // 64}
    batch = MR.make_batch(B, T, n_img_tok, 224, seed=1)
    wkv = MR.oracle_wkv("f32")

    def step():
        for t in P.values():
            t.grad = None
        logits, targets = MR.visual_forward(P, batch, cfg, wkv)
        loss = MR.training_loss(logits, targets)
        loss.backward()
        return float(loss)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    try:
        import cpuinfo  # py_cpuinfo
        cpu_name = cpuinfo.get_cpu_info().get("brand_raw", "unknown")
    except Exception:
        cpu_name = "unknown"
    return {"value": B * T / dt, "unit": "tokens/s", "cores": ncores, "kind": "port", "cpu": cpu_name,
            "sample": f"fwd+bwd of the same 0.1B+SigLIP-B/16 model, fp32, B={B} T={T} ({n_img_tok} image tokens), "
                      f"{steps} steps after {warmup} warm-up, torch CPU + C oracle WKV7 (OpenMP)",
            "ms_per_step": dt * 1e3}


def ref_kernel_times(B, T, H, dev):
    """ms per launch of the reference forward_kernel / backward_kernel (wkv7_cuda.cu) on (B,T,H,64) realistic inputs;
    None when oracle/_ref was not built (no /root/reference at build time)."""
    try:
        from oracle import ref_kernel as RK
        from oracle import wkv7 as O
        if not RK.available():
            return None
        inp = [x.to(dev) for x in O.make_inputs(B, T, H, 64, seed=42)]
        out = {}
        for name, fn in (("fwd", lambda: RK.forward(*inp[:6])), ("bwd", None)):
            if name == "bwd":
                _, rs, rsa = RK.forward(*inp[:6])
                fn = lambda: RK.backward(*inp, rs, rsa)  # noqa: E731
            for _ in range(2):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                fn()
            e1.record()
            torch.cuda.synchronize()
            out[name] = e0.elapsed_time(e1) / 5
        return out
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:200]}


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS), help="BASELINE.json configs[1] (headline) or configs[2]")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the config's)")
    ap.add_argument("--ctx", type=int, default=None)
    ap.add_argument("--layers", type=int, default=None)
    ap.add_argument("--embd", type=int, default=None)
    ap.add_argument("--wkv", default="x6", choices=sorted(WKV_PATHS),
                    help="WKV7 kernels of the time-mix block: x6 (default; chunked tensor-core kernels at fp32-level accuracy, pass the "
                         "strict parity tests), step (step-by-step fp32 kernels), tf32 (round-1 kernels, outside the tolerance)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step as one CUDA graph (visualrwkv_b200.graph.GraphedTrainStep); auto = on")
    ap.add_argument("--optimizer", default="own", choices=["own", "torch"],
                    help="own: visualrwkv_b200.optim.FusedAdamW (one multi-tensor kernel); torch: stock fused AdamW on fp32 copies")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-kernel", action="store_true")
    ap.add_argument("--grad-cp", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss and a fixed sample of every trainable parameter's gradient and "
                         "updated value from the last timed step to DIR/*.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[a.config]
    for k_ in ("batch", "ctx", "layers", "embd"):
        if getattr(a, k_) is None:
            setattr(a, k_, cfg[k_])

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": f"{cfg['name']} + SigLIP-B/16@224 (196 patches -> AdaptiveAvgPool -> 576 image tokens), "
                          f"ctx {a.ctx}, batch {a.batch}/GPU, fwd+bwd+allreduce+AdamW; WKV7 path: {a.wkv}",
              "global_batch": a.batch * world, "seq_len": a.ctx, "image_tokens": 576, "parallelism": f"dp{world}", "wkv": a.wkv,
              "l2": "working set per step (>2 GB of activations) exceeds the 126 MB L2; no explicit flush"}

    if a.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(max(a.steps, 1), a.warmup)
        config["reference_sample"] = r["sample"]   # what one timed step of this arm actually is (a bounded sample of the workload)
        line = {"impl": "reference", "metric": "tokens/s fwd+bwd (T=2048, 576 img-tok)", "value": r["value"], "unit": "tokens/s",
                "n_gpus": a.gpus, "steps": max(a.steps, 1), "warmup": a.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu")},
                "e2e": {"value": r["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py (impl ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from visualrwkv_b200 import _lib, fused, wkv7
    fused.set_wkv_path(a.wkv)
    from visualrwkv_b200.benchutil import ClockSampler
    from visualrwkv_b200.ddp import GradBucketReducer
    from visualrwkv_b200.model import VisualRWKV, default_args, randomize_zero_init
    from visualrwkv_b200.synthetic import make_batch
    _lib.load_torch_ops()

    torch.manual_seed(1234)
    args = default_args(n_layer=a.layers, n_embd=a.embd, dim_att=a.embd, ctx_len=a.ctx, grad_cp=a.grad_cp)
    model = VisualRWKV(args)
    randomize_zero_init(model)
    model = model.to(device=dev, dtype=torch.bfloat16)
    model.freeze_emb()  # v7.00/train.py:196: emb is always frozen
    trainable = [p for p in model.parameters() if p.requires_grad]
    reducer = GradBucketReducer(trainable) if world > 1 else None
    # bf16 params + fp32 master/Adam state (what DeepSpeed bf16 keeps): one multi-tensor AdamW kernel (csrc/optim.cu);
    # --optimizer torch: stock PyTorch (bf16 -> fp32 gradient copy, fused AdamW on fp32 copies, copy back)
    use_graph = a.graph != "off"
    if a.optimizer == "own":
        from visualrwkv_b200.optim import FusedAdamW
        opt = FusedAdamW(trainable, lr=1e-5, betas=(0.9, 0.99), eps=1e-8, weight_decay=0.0)
        master = None
    else:
        master = [p.detach().float().clone() for p in trainable]
        for mp in master:
            mp.grad = torch.zeros_like(mp)
        opt = torch.optim.AdamW(master, lr=torch.tensor(1e-5, device=dev) if use_graph else 1e-5, betas=(0.9, 0.99), eps=1e-8,
                                weight_decay=0.0, fused=True, capturable=use_graph)

    B, T = a.batch, a.ctx
    host = make_batch(B, T, 576, 224, seed=100 + rank, img_dtype=torch.bfloat16)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    resident = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))

    def apply_grads_local():
        with torch.no_grad():
            if master is None:
                opt.step()
            else:
                torch._foreach_copy_([m.grad for m in master], [p.grad for p in trainable])
                opt.step()
                torch._foreach_copy_(trainable, master)

    def apply_grads():
        if reducer is not None:
            reducer.finish()
        apply_grads_local()

    def eager_step(batch):
        if reducer is not None:
            reducer.reset()
        else:
            for p in trainable:
                p.grad = None
        loss = model.training_step(batch)
        loss.backward()
        apply_grads()
        return loss

    train_step = eager_step
    graph_note = "eager launches"
    if use_graph:
        try:
            from visualrwkv_b200.graph import GraphedTrainStep
            if reducer is None:
                gstep = GraphedTrainStep(model, resident, after_backward=apply_grads)
                train_step = gstep
                graph_note = "one CUDA graph per step (forward + backward + AdamW)"
            else:
                # collectives stay outside the graphs (NCCL inside a capture hung on this stack): graph 1 = forward + backward into
                # the flat gradient buckets, then one NCCL all-reduce per bucket, then graph 2 = master copy + AdamW + copy back
                reducer.overlap = False
                gstep = GraphedTrainStep(model, resident, before_forward=reducer.zero_buckets, set_grads_to_none=False)
                opt_graph = torch.cuda.CUDAGraph()
                reducer.allreduce_all()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    apply_grads_local()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                with torch.cuda.graph(opt_graph):
                    apply_grads_local()

                def graphed_ddp_step(batch):
                    loss = gstep(batch)
                    reducer.allreduce_all()
                    opt_graph.replay()
                    return loss

                train_step = graphed_ddp_step
                graph_note = "CUDA graph (forward + backward) + NCCL all-reduce per bucket + CUDA graph (AdamW)"
        except Exception as e:  # noqa: BLE001
            if a.graph == "on":
                raise
            graph_note = f"eager launches (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
            if reducer is not None:
                reducer.overlap = True
            train_step = eager_step
            torch.cuda.synchronize()
    config["launch"] = graph_note
    config["optimizer"] = "AdamW, fp32 master + moments, " + ("one multi-tensor kernel (csrc/optim.cu)" if a.optimizer == "own"
                                                                else "torch fused AdamW on fp32 copies")

    def e2e_step():
        if train_step is not eager_step:
            loss = train_step(host)   # the graphed step copies the pinned host tensors into its static device buffers (H2D)
        else:
            batch = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in host.items()}
            loss = train_step(batch)
        return float(loss.detach())  # D2H read of the loss (synchronises)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    graphed = train_step is not eager_step
    for _ in range(max(a.warmup, 3)):
        train_step(resident)
    if not graphed:
        wkv7.PROFILE = []
    lc0 = wkv7.launch_count()
    last = {}

    def timed_step():
        last["loss"] = train_step(resident)

    with ClockSampler(local_rank) as cs:
        ms = timed(timed_step, a.steps)
    launches = wkv7.launch_count() - lc0
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, last["loss"], [(n, p) for n, p in model.named_parameters() if p.requires_grad])
    if graphed:
        # a replayed graph does not pass through the host-side launch counter, and CUDA events cannot time single kernels
        # inside it: count the launches of ONE eager replica of the step and time the WKV7 kernels there (same kernels,
        # same shapes, same buffers), right after the timed region
        torch.cuda.synchronize()
        eager_step(resident)
        wkv7.PROFILE = []
        lc0 = wkv7.launch_count()
        eager_step(resident)
        eager_step(resident)
        launches = (wkv7.launch_count() - lc0) // 2 * a.steps
    prof, wkv7.PROFILE = wkv7.PROFILE, None
    prof_steps = 2 if graphed else a.steps
    torch.cuda.synchronize()
    ms_e2e = timed(e2e_step, a.steps)

    tokens = B * T * world
    value = tokens / (ms / 1e3)
    line = {"metric": "tokens/s fwd+bwd (T=2048, 576 img-tok)", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
            "e2e": {"value": tokens / (ms_e2e / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e},
            "gpu_launches": launches, "tokens_per_s_per_gpu": value / world, "clocks": cs.summary()}

    if rank == 0:
        peaks = load_peaks()
        nel = B * T * args.n_embd
        fwd = [e0.elapsed_time(e1) for kind, e0, e1 in prof if kind == "fwd"]
        bwd = [e0.elapsed_time(e1) for kind, e0, e1 in prof if kind == "bwd"]
        if fwd and bwd:
            fms, bms = sum(fwd) / len(fwd), sum(bwd) / len(bwd)
            peak = peaks["hbm_gbs"]
            # DRAM bytes per launch from the ncu --set full capture of this configuration (profiles/r1e_wkv7_tc_model_path_summary.csv)
            wp = WKV_PATHS[a.wkv]
            at_cfg2 = (B, T, args.n_embd) == (8, 2048, 768)
            line["roofline"] = {"kernel": "wkv7 backward = " + wp["bwd"], "bound": "hbm", "achieved": WKV_BWD_BYTES_PER_ELEM * nel / bms / 1e6,
                                "peak": peak, "unit": "GB/s", "frac": WKV_BWD_BYTES_PER_ELEM * nel / bms / 1e6 / peak,
                                "traffic": wp["traffic_bwd"] if at_cfg2 else None, "traffic_unit": "bytes", "traffic_source": wp["ncu"],
                                "avg_launch_ms": bms, "launches_timed": len(bwd),
                                "peak_source": peaks["source"], "share_of_step": sum(bwd) / prof_steps / ms,
                                "timed_in": "eager replica of the step right after the timed region (the timed region replays one CUDA graph)" if graphed else "the timed region"}
            line["roofline_wkv7_fwd"] = {"kernel": wp["fwd"], "bound": "hbm", "achieved": WKV_FWD_BYTES_PER_ELEM * nel / fms / 1e6,
                                         "peak": peak, "unit": "GB/s", "frac": WKV_FWD_BYTES_PER_ELEM * nel / fms / 1e6 / peak,
                                         "traffic": wp["traffic_fwd"] if at_cfg2 else None,
                                         "traffic_unit": "bytes", "avg_launch_ms": fms, "launches_timed": len(fwd),
                                         "share_of_step": sum(fwd) / prof_steps / ms}
        # model FLOPs (GEMMs only, SURVEY.md §8d): fwd 281 MFLOP/token at 0.1B -> x3 for fwd+bwd
        C, L, V = args.n_embd, args.n_layer, args.vocab_size
        lora = LORA_RANKS.get(C, 0)
        per_tok = L * (8 * C * C + 4 * C * lora + 16 * C * C) + 2 * C * V
        line["gemm_tflops_achieved"] = 3 * per_tok * B * T / (ms / 1e3) / 1e12
        line["gemm_frac_of_bf16_peak"] = line["gemm_tflops_achieved"] / (peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"])
        if world == 1 and not a.no_ref_kernel:
            # the reference's own WKV7 kernel (oracle/_ref, compiled from the mounted sources) on the same GPU and inputs,
            # outside the timed region: makes the "x reference kernel" figures driver-observable
            rk = ref_kernel_times(B, T, args.dim_att // 64, dev)
            if rk is not None:
                line["ref_kernel_ms"] = rk
                if fwd and bwd:
                    line["wkv7_speedup_vs_ref_kernel"] = {"fwd": rk["fwd"] / fms, "bwd": rk["bwd"] / bms}
        if world == 1 and not a.no_cpu_baseline:
            r = cpu_reference_run(steps=3, warmup=1)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu")}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
