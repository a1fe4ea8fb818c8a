#!/usr/bin/env python
"""bench.py - 256^2 perceptual-loss training images/sec (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus 1 --steps K --warmup W              # our arm (libast_b200.so kernels)
  torchrun --nproc-per-node N ... bench.py --gpus N ...       # data-parallel, one rank per GPU, NCCL allreduce
  python bench.py --impl reference ...                        # the reference's CPU step (oracle port) on host cores

A "step" is one full optimisation step of train_cnn.py:295-334 (TransformerNet fwd/bwd, VGG taps, Grams,
style/content MSE, gradient all-reduce, Adam) on one synthetic batch.  Workload at every N: BASELINE
configs[1] - batch 32 per GPU at 256x256, bf16-in/fp32-accumulate ("fast" precision) - weak scaling.
Prints ONE JSON line (rank 0).

Roofline numbers: per-kernel device durations come from the CUDA-GRAPH REPLAY of the step (CUPTI through
torch.profiler over 3 replays, taken AFTER the timed region - the headline value is never measured under a
profiler), so the family times sum to the step time; algorithmic flops / bytes per family come from the
library's own launch accounting (ast_family_stats) over one eager step of the same workload.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md 8(d): algorithmic work per training image at 256^2 (scales with H*W)
GF_PER_IMG = {"total": 137.86, "conv_gather": 16.803 + 15.784 + 36.465 + 36.465 + 12.306 + 2.147,
              "wgrad_gather": 16.803, "gram": 1.082}
IN_ELEMS_PER_IMG = 13.107e6   # elements through the 17 InstanceNorm layers at 256^2
CONV_FAMILIES = ("conv_hx", "conv_st", "conv_px", "conv_ws", "conv_tc", "conv_simt")


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "src": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "B200_PROFILING.md fallback"}


def read_traffic():
    """DRAM bytes per launch of each kernel family from the committed ncu --set full captures (profiles/r02_traffic.json,
    written by profiles/summarize_ncu.py from the raw CSVs next to it); absent -> null in the JSON line."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    return json.load(open(path)) if os.path.exists(path) else {}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.idx = None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        """Median SM clock / throttle reasons of the samples whose timestamp falls inside [t_begin, t_end] (the sampler
        is started before the warm-up so that it is already streaming when the timed region begins)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        import datetime
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, mxv = float(f[1]), float(f[2])
            except ValueError:
                continue
            if t_begin is not None and not (t_begin - 0.03 <= ts <= t_end + 0.03):
                continue
            sm.append(clk); mx = mxv
            try:
                power.append(float(f[3]))
            except ValueError:
                pass
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


def cpu_reference_step_rate(batch, size, steps, warmup, threads):
    """The reference's training step (oracle port of train_cnn.py:295-334 + Adam) on the host cores."""
    import torch
    from oracle import port, weights
    torch.set_num_threads(threads)
    tsd = port.make_leaf(weights.transfer_state_dict(2), torch.float32)
    vsd = weights.vgg_state_dict(2)
    style = port.style_grams_single(weights.style_image(size, 2), vsd, batch)
    state, params = {}, tsd
    times = []
    for it in range(warmup + steps):
        content = weights.content_batch(batch, size, 2, step=it)
        t0 = time.perf_counter()
        leaf = port.make_leaf(params, torch.float32)
        out = port.training_step(leaf, vsd, content, style)
        params = port.adam_l2_step({k: v.detach() for k, v in leaf.items()}, out["grads"], state, 0.0024, it + 1)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return batch * len(times) / sum(times), sum(times) / len(times) * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    batch = 4
    rate, ms = cpu_reference_step_rate(batch, args.size, args.steps, args.warmup, threads)
    sample = f"B={batch} images of {args.size}x{args.size} per step, fp32, torch CPU ops, {threads} threads"
    line = {"impl": "reference", "metric": "train_images_per_sec_256", "value": rate, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"perceptual-loss training step, {args.size}x{args.size}, CPU sample of B={batch} "
                                   "(BASELINE configs[1] is B=32/GPU)"},
            "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def kernel_family(name):
    """Kernel name (as CUPTI reports it) -> family of ast_family_stats, or 'torch/other' for anything not ours."""
    if "ast::" not in name and "fold_rows" not in name:
        return "nccl" if "nccl" in name.lower() else "torch/other"
    for key, fam in (("conv_hx_kernel", "conv_hx"), ("conv_st_kernel", "conv_st"), ("conv_px_kernel", "conv_px"), ("conv_ws_kernel", "conv_ws"), ("conv_tc_kernel", "conv_tc"),
                     ("conv_gather_simt", "conv_simt"), ("contract_thin", "wgrad_thin"),
                     ("contract_tc_kernel<0>", "wgrad_tc"), ("contract_tc_kernel<1>", "gram_tc"),
                     ("contract_tc_kernel<(int)0>", "wgrad_tc"), ("contract_tc_kernel<(int)1>", "gram_tc"),
                     ("wgrad_gather_simt", "wgrad_simt"), ("in_apply", "in_apply"), ("in_bwd", "in_bwd"),
                     ("in_finalize", "in_stats"), ("in_stats", "in_stats"), ("maxpool", "pool"), ("mse", "mse"),
                     ("gram_finish", "mse"), ("adam", "optim"), ("batch_reduce", "optim"), ("pack_weights", "optim")):
        if key in name:
            return fam
    return "pointwise"


def profile_replays(step_fn, replays):
    """{kernel name: (ms per step, launches per step)} of `replays` calls of step_fn (graph replays), via CUPTI."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(replays):
            step_fn()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0.0, 0])
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            t = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
            agg[ev.name][0] += t / 1e3 / replays
            agg[ev.name][1] += 1.0 / replays
    return {k: (v[0], v[1]) for k, v in agg.items()}


def timed(fn, reps, warm=1):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def other_configs(ast, dist, dev, rank, world, peaks):
    """Short legs for BASELINE configs[2..4] (not the headline): smartaverage over 512^2 paintings (sharded over the
    ranks with the C2 all-reduce when world > 1), 1080p stylisation B=8 through the fused uint8 boundary, 1024^2 step."""
    import torch
    out = {}
    torch.manual_seed(2)
    net = ast.StyleTransfer(device=dev, precision="fast")
    vgg = ast.VGG16(vgg_path=None, precision="fast").to(dev)
    peak = peaks["bf16_tflops_sustained"]
    # ---- configs[2]: 'smartaverage', 512^2, 16 paintings per rank (the real job: 4096 / 8 = 512 per rank)
    per_rank = 16
    g = torch.Generator(device=dev).manual_seed(2 + rank)
    paint = [torch.randint(0, 256, (3, 512, 512), device=dev, generator=g).float() for _ in range(per_rank)]
    grp = dist.group.WORLD if world > 1 else None
    for mode in ("reference", "mean_gram"):
        ms = timed(lambda: ast.style_grams_smartaverage(vgg, paint, 1, mode=mode, group=grp), 2)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        rate = per_rank * world / (ms / 1e3)
        out[f"config3_smartaverage_{mode}"] = {
            "value": rate, "unit": "paintings/s", "ms": ms, "paintings": per_rank * world,
            "allreduce_bytes_per_rank": (31.46e6 * 4 if mode == "reference" else 1.39e6),
            "tensor_frac": 145.86 * rate / world / 1e3 / peak}
    del paint
    # ---- configs[3]: 1080p stylisation, batch 8, uint8 BGR in -> uint8 RGB out (inference.py:107-116 fused)
    x = torch.randint(0, 256, (8, 1080, 1920, 3), device=dev, dtype=torch.uint8)
    y = net.stylize(x)
    assert y.shape == x.shape and y.dtype == torch.uint8
    ms = timed(lambda: net.stylize(x), 3)
    out["config4_1080p_stylize_b8"] = {"value": 8 * world / (ms / 1e3), "unit": "images/s", "ms": ms,
                                       "tensor_frac": 531.64 * 8 / ms / peak, "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9}
    del x, y
    torch.cuda.empty_cache()
    # ---- configs[4]: 1024^2 training step, batch 4 per GPU
    style = ast.style_grams_single(vgg, torch.randint(0, 256, (3, 1024, 1024), device=dev).float(), 4)
    tr = ast.PerceptualTrainer(net, vgg, style)
    xb = torch.randint(0, 256, (4, 3, 1024, 1024), device=dev, dtype=torch.uint8)
    ms = timed(lambda: tr.step(xb), 3, warm=2)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    out["config5_1024_step_b4"] = {"value": 4 * world / (ms / 1e3), "unit": "images/s", "ms": ms,
                                   "tensor_frac": 2205.7 * 4 / ms / peak}
    tr.close()
    return out


def dp_check(ast, dist, dev, rank, world):
    """Data-parallel exactness (SURVEY 8e) checked on the NCCL path before timing: the mean of the per-rank losses and
    the all-reduced gradient arena of `world` shards of 4 images == one pass over the 4*world images on rank 0."""
    import torch
    torch.manual_seed(2)
    net = ast.StyleTransfer(device=dev, precision="fast")
    vgg = ast.VGG16(vgg_path=None, precision="fast").to(dev)
    bs, S = 4, 128
    full = torch.randint(0, 256, (bs * world, 3, S, S), device=dev, generator=torch.Generator(device=dev).manual_seed(5)).float()
    style_img = torch.randint(0, 256, (3, S, S), device=dev, generator=torch.Generator(device=dev).manual_seed(6)).float()
    arena = net._arena_for(dev)
    gbuf = arena.new_grad_buffer()
    arena.grad_sink = gbuf
    # sharded: this rank's 4 images, gradients averaged over ranks through the trainer's own all-reduce path
    style = ast.style_grams_single(vgg, style_img, bs)
    c, s, t = ast.perceptual_step(net, vgg, full[rank * bs:(rank + 1) * bs], style)
    from artist_style_transfer_b200 import dp
    dp.allreduce_mean_flat(gbuf, None)
    losses = torch.stack([c, s, t])
    dist.all_reduce(losses, op=dist.ReduceOp.AVG)
    sharded = gbuf.clone()
    res = None
    if rank == 0:
        gbuf.zero_()
        style_full = ast.style_grams_single(vgg, style_img, bs * world)
        c2, s2, t2 = ast.perceptual_step(net, vgg, full, style_full)
        ref = torch.stack([c2, s2, t2])
        loss_rel = float(((losses - ref).abs() / ref.abs()).max())
        grad_rel = float((sharded - gbuf).norm() / gbuf.norm())
        res = {"loss_rel": loss_rel, "grad_rel": grad_rel, "images": bs * world, "size": S,
               "ok": bool(loss_rel < 2e-3 and grad_rel < 3e-2)}
    arena.grad_sink = None
    # C2: 'smartaverage' sharded over the ranks (each rank its paintings, one all-reduce of the sums) == all paintings on one rank
    paint = [torch.randint(0, 256, (3, S, S), device=dev, generator=torch.Generator(device=dev).manual_seed(40 + i)).float()
             for i in range(2 * world)]
    lo, hi = dp.shard_range(len(paint), rank, world)
    for mode in ("reference", "mean_gram"):
        sharded_g = ast.style_grams_smartaverage(vgg, paint[lo:hi], 1, mode=mode, group=dist.group.WORLD)
        if rank == 0:
            seq = ast.style_grams_smartaverage(vgg, paint, 1, mode=mode)
            err = max(float((sharded_g[k] - seq[k]).norm() / seq[k].norm()) for k in seq)
            res[f"smartaverage_{mode}_rel"] = err
            res["ok"] = bool(res["ok"] and err < 1e-4)
    torch.cuda.synchronize()
    dist.barrier()
    return res


def run_ours(args):
    # keep stdout clean for the ONE JSON line: libraries (e.g. "NCCL version ...") write to fd 1 during init
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch
    import torch.distributed as dist
    import artist_style_transfer_b200 as ast
    from artist_style_transfer_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B, S, K, W = args.batch, args.size, args.steps, args.warmup
    in_dtype = torch.uint8 if args.input == "uint8" else torch.float32

    check = dp_check(ast, dist, dev, rank, world) if world > 1 else None
    if check is not None and not check["ok"]:
        raise SystemExit(f"data-parallel equivalence check failed, not timing a wrong step: {check}")

    torch.manual_seed(2 + rank)                            # replicas are made identical by the trainer's broadcast
    net = ast.StyleTransfer(device=dev, precision=args.precision)
    vgg = ast.VGG16(vgg_path=None, precision=args.precision).to(dev)
    if world > 1:                                          # the frozen VGG is not a trained parameter: same on all ranks
        for p in vgg.parameters():
            dist.broadcast(p.data, src=0)
    gen = torch.Generator(device=dev).manual_seed(2 + 7919 * rank)
    style_img = torch.randint(0, 256, (3, S, S), device=dev, generator=torch.Generator(device=dev).manual_seed(2)).float()
    style = ast.style_grams_single(vgg, style_img, B)
    trainer = ast.PerceptualTrainer(net, vgg, style, cuda_graph=not args.no_graph)
    nbuf = 4
    batches = [torch.randint(0, 256, (B, 3, S, S), device=dev, generator=gen).to(in_dtype) for _ in range(nbuf)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(W + (4 if not args.no_graph else 0)):   # graph mode: 3 eager steps + capture happen before timing
        trainer.step(batches[i % nbuf])
    barrier()
    t_begin = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        losses = trainer.step(batches[i % nbuf])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t_begin, time.time()) if rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = B * world * K / (ms / 1e3)
    losses_last = [float(x) for x in losses]

    # ---- e2e: pinned host buffers -> H2D copy -> step -> D2H loss read, every step (same workload, --steps steps)
    host = [torch.randint(0, 256, (B, 3, S, S)).to(in_dtype).pin_memory() for _ in range(2)]
    loss_host = torch.zeros(3, dtype=torch.float32).pin_memory()
    ke = K
    for i in range(2):                                      # untimed: staging buffers / pinned pages are touched once
        trainer.step(trainer.prefetch(host[i]))
    barrier()
    e0.record()
    nxt = trainer.prefetch(host[0])                         # H2D of step 0's inputs (inside the timed region)
    for i in range(ke):
        x = nxt
        if i + 1 < ke:                                      # public API: the next batch's H2D copy runs on a side stream
            nxt = trainer.prefetch(host[(i + 1) % 2])       # while this step computes; every step still copies its inputs
        c, s, tot = trainer.step(x)
        loss_host.copy_(torch.stack([c, s, tot]), non_blocking=True)
        torch.cuda.current_stream().synchronize()           # the caller reads the loss
    e1.record()
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = B * world * ke / (float(te.item()) / 1e3)

    # ---- algorithmic work per kernel family: the library's accounting over ONE eager step of the same workload
    lc0, fs0 = _lib.launch_count(), _lib.family_stats()
    trainer._eager_step(batches[0], trainer.style_gram)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - lc0
    work = _lib.family_delta(fs0)
    # ---- device time per kernel from the graph replay (CUPTI, after the timed region)
    R = 3
    kern = profile_replays(lambda: trainer.step(batches[0]), R)
    fam_ms, fam_n = collections.defaultdict(float), collections.defaultdict(float)
    for name, (kms, cnt) in kern.items():
        fam_ms[kernel_family(name)] += kms
        fam_n[kernel_family(name)] += cnt
    sum_ms = sum(fam_ms.values())

    peaks = read_peaks()
    traffic = read_traffic()
    scale = (S / 256.0) ** 2
    peak_tf, peak_bw = peaks["bf16_tflops_sustained"], peaks["hbm_gbs"]
    # TF32 peak is not in MEASURED_PEAKS.json (BASELINE.md section 5): measured here the same way (cuBLAS 8192^3, best of 6)
    tf32_peak = None
    if rank == 0 and args.precision == "fast":
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a_ = torch.randn(8192, 8192, device=dev); b_ = torch.randn(8192, 8192, device=dev)
        best = 1e9
        for _ in range(6):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); torch.matmul(a_, b_); t1.record(); torch.cuda.synchronize()
            best = min(best, t0.elapsed_time(t1))
        tf32_peak = 2 * 8192 ** 3 / best / 1e9
        torch.backends.cuda.matmul.allow_tf32 = old
        del a_, b_

    def entry(fam, bound, algo, unit_peak):
        ms_f = fam_ms.get(fam, 0.0)
        if ms_f <= 0:
            return None
        achieved = algo / (ms_f / 1e3) / (1e12 if bound == "tensor" else 1e9)
        tr = traffic.get(fam)
        return {"kernel": fam, "bound": bound, "achieved": achieved, "peak": unit_peak,
                "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": achieved / unit_peak,
                "ms_per_step": ms_f, "launches_per_step": fam_n.get(fam, 0.0),
                "launch_ms_avg": ms_f / max(1.0, fam_n.get(fam, 1.0)),
                "algorithmic_per_step": algo, "traffic": None if not tr else tr.get("dram_bytes_per_launch"),
                "traffic_src": None if not tr else tr.get("src")}

    # conv families: the library counts executed flops (3-channel ends padded to 32); scale them so that all conv launches
    # together carry SURVEY 8(d)'s algorithmic 119.97 GF per image
    lib_conv = sum(work[f][1] for f in CONV_FAMILIES if f in work)
    conv_algo_total = GF_PER_IMG["conv_gather"] * 1e9 * scale * B
    rooflines = []
    for f in CONV_FAMILIES:
        if f in work and work[f][1] > 0:
            rooflines.append(entry(f, "tensor", work[f][1] / lib_conv * conv_algo_total, peak_tf))
    wg = sum(work[f][1] for f in ("wgrad_tc", "wgrad_thin", "wgrad_simt") if f in work)
    for f in ("wgrad_tc", "wgrad_thin", "wgrad_simt"):
        if f in work and work[f][1] > 0:
            rooflines.append(entry(f, "tensor", work[f][1] / wg * GF_PER_IMG["wgrad_gather"] * 1e9 * scale * B, peak_tf))
    for f in ("gram_tc", "gram_simt"):                     # Gram at 256^2 is HBM bound (SURVEY 8a): one read of F + G out
        if f in work and work[f][2] > 0:
            rooflines.append(entry(f, "hbm", work[f][2], peak_bw))
    for f in ("in_apply", "in_bwd", "pool", "mse", "pointwise", "optim"):
        if f in work and work[f][2] > 0:
            rooflines.append(entry(f, "hbm", work[f][2], peak_bw))
    rooflines = [r for r in rooflines if r]
    conv_ms = sum(fam_ms.get(f, 0.0) for f in CONV_FAMILIES)
    conv_tf = conv_algo_total / (conv_ms / 1e3) / 1e12
    # kind::tf32: only the Gram backward (2.147 GF/img; its F operand is an fp32 tap).  kind::f16: TransformerNet forward /
    # dgrad and the VGG dgrad in bf16, the VGG forward (36.465 + 12.306) with fp16 operands - the 10 mantissa bits TF32
    # keeps of an fp32 value, at the 16-bit MMA rate.
    tf32_share = 2.147 / GF_PER_IMG["conv_gather"]
    mix_peak = None if not tf32_peak else 1.0 / (tf32_share / tf32_peak + (1 - tf32_share) / peaks["bf16_tflops"])
    roofline_conv = {"kernel": "all conv fwd/dgrad launches of one step (conv_hx + conv_st + conv_px + conv_ws + conv_tc kernels)",
                     "bound": "tensor", "achieved": conv_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": conv_tf / peak_tf,
                     "ms_per_step": conv_ms, "peak_source": f"{peaks['src']} bf16 sustained",
                     "tf32_tflops_measured_here_cublas_8192": tf32_peak, "tf32_flop_share": tf32_share,
                     "frac_of_precision_mix_peak": None if not mix_peak else conv_tf / mix_peak, "traffic": None}
    esz = 2 if args.precision == "fast" else 4
    in_ms = fam_ms.get("in_apply", 0.0) + fam_ms.get("in_bwd", 0.0) + fam_ms.get("in_stats", 0.0)
    in_gb = IN_ELEMS_PER_IMG * scale * B * esz * 5 / 1e9                 # fwd 1R+1W, bwd 2R+1W
    tr_in = traffic.get("in_bwd")
    roofline_in = {"kernel": "InstanceNorm (in_apply_staged fwd; in_bwd_* bwd; forward statistics ride in the conv epilogues)",
                   "bound": "hbm", "achieved": in_gb / (in_ms / 1e3), "peak": peak_bw, "unit": "GB/s",
                   "frac": in_gb / (in_ms / 1e3) / peak_bw, "ms_per_step": in_ms,
                   "traffic": None if not tr_in else tr_in.get("dram_bytes_per_launch"),
                   "note": "13.107 M elements/img x 5 algorithmic passes (SURVEY 8d)"}
    dominant = max(rooflines, key=lambda r: r["ms_per_step"]) if rooflines else roofline_conv
    dominant = dict(dominant, peak_source=f"{peaks['src']} ({'bf16 sustained' if dominant['bound'] == 'tensor' else 'HBM copy'})")

    extra = None
    if not args.no_other_configs:
        trainer.close()
        del trainer, batches, host
        torch.cuda.empty_cache()
        extra = other_configs(ast, dist, dev, rank, world, peaks)
        trainer = None
    if trainer is not None:
        trainer.close()
    if world > 1:                      # everyone is done with the GPU work; from here on only rank 0 has something to do
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        rate, _ = cpu_reference_step_rate(4, S, 3, 1, threads)
        cpu_baseline = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                        "sample": f"1 warm-up + 3 timed steps of B=4 at {S}x{S}, fp32 oracle port of train_cnn.py:295-334 + Adam"}
    in_bytes = B * 3 * S * S * (1 if in_dtype == torch.uint8 else 4)
    line = {
        "metric": "train_images_per_sec_256", "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "fast" else "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[1]: perceptual-loss training step, {S}x{S}, batch {B}/GPU, "
                               f"precision={args.precision}, random-init TransformerNet+VGG16, fused Adam(L2)",
                   "global_batch": B * world, "parallelism": f"dp{world}", "cuda_graph": not args.no_graph,
                   "input": f"{args.input} BGR [B,3,{S},{S}] (dataset.py:97-108 images are uint8-derived)",
                   "l2": "per-step working set (GBs of activations) >> 126 MB L2; inputs rotate over 4 buffers",
                   "arithmetic": ("TransformerNet + VGG gradient chain bf16, VGG forward fp16 operands (10-bit mantissa, the "
                                  "precision of TF32) with fp32 taps, Grams TF32; fp32 accumulation everywhere"
                                  if args.precision == "fast" else "fp32 FFMA")},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 12, "steps": ke},
        "gpu_launches": int(launches_per_step * K), "gpu_launches_per_step": int(launches_per_step), "clocks": clocks,
        "roofline": dominant, "roofline_conv": roofline_conv, "roofline_instnorm": roofline_in, "rooflines": rooflines,
        "family_ms_per_step": dict(fam_ms), "sum_kernel_ms_per_step": sum_ms,
        "timing_source": f"CUPTI kernel durations over {R} CUDA-graph replays after the timed region",
        "cpu_baseline": cpu_baseline, "dp_check": check, "other_configs": extra,
        "losses_last_step": losses_last,
        "gflop_per_image": GF_PER_IMG["total"] * scale,
        "tensor_frac_whole_step": GF_PER_IMG["total"] * scale * B * K / ms / peak_tf,
    }
    if args.dump_outputs:
        # what trainer.step() returned in the last timed step.  The updated parameters are not written: Adam turns the
        # last-bit differences of reordered sums into lr-sized steps: two runs of the same build at the default arguments
        # ended 5-20 % apart in each conv weight while their losses agreed to 6e-4 (one B200 at 1000 W).
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "losses.npy"), np.array(losses_last, dtype=np.float64))
    os.write(json_fd, (json.dumps(line) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--batch", type=int, default=32, help="images per GPU per step")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--input", default="uint8", choices=["uint8", "float32"], help="dtype of the content batches")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short BASELINE configs[2..4] legs")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's [content, style, total] losses to DIR/losses.npy (inputs and "
                         "initial weights are seeded, so runs with the same arguments can be compared)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
