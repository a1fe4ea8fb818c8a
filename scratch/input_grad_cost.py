"""Cost of the input gradient of the TransformerNet modules (fast mode, B200).

Times, alternating the variants in every repetition (CUDA events, one forward + backward per call):
  - StyleTransfer forward + backward at B=32, 256^2 with and without x.requires_grad_();
  - the same network rebuilt as an nn.Sequential of its standalone modules (every module one autograd node, so every
    module's input gradient runs) against the fused module;
and, in a separate profiled pass, the launches that only the input-gradient variant issues (the stage-0 data gradient,
its on-demand pack, ast_reflect_fold) with the achieved bandwidth of ast_reflect_fold.  The device name and power limit
are printed with the numbers.  Usage: python scratch/input_grad_cost.py [--batch 32] [--size 256] [--reps 5] [--iters 10]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

import artist_style_transfer_b200 as ast  # noqa: E402
from artist_style_transfer_b200 import ops  # noqa: E402
from oracle import weights  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return f"{torch.cuda.get_device_name()} | nvidia-smi: {q[torch.cuda.current_device()] if q else 'n/a'}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    dev = torch.device("cuda")
    net = ast.StyleTransfer(device=dev, precision="fast")
    net.load_state_dict(weights.transfer_state_dict(2), strict=True)
    seq = nn.Sequential(*net.ConvBlock, *net.ResidualBlock, *net.DeconvBlock)     # same parameters, one node per module
    for m in seq.modules():
        if hasattr(m, "precision"):
            m.precision = "fast"
    x = weights.content_batch(a.batch, a.size, 2).to(dev)
    xg = x.clone().requires_grad_(True)
    gy = torch.randn(a.batch, 3, a.size, a.size, device=dev)

    def run(module, inp):
        module.zero_grad(set_to_none=True)
        inp.grad = None
        module(inp).backward(gy)

    variants = {"fused, x without grad": lambda: run(net, x), "fused, x.requires_grad_()": lambda: run(net, xg),
                "Sequential of modules, x without grad": lambda: run(seq, x)}
    for fn in variants.values():                        # warm-up: packs, tap tables, allocator
        fn()
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(a.reps):
        for name, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / a.iters)
    print(f"device: {device_info()}")
    print(f"StyleTransfer forward + backward, fast mode, B={a.batch}, {a.size}^2, {a.reps} alternating repetitions of "
          f"{a.iters} calls (ms per call: median [min, max])")
    base = sorted(times["fused, x without grad"])[a.reps // 2]
    for name, t in times.items():
        t = sorted(t)
        print(f"  {name:40s} {t[a.reps // 2]:8.3f} [{t[0]:.3f}, {t[-1]:.3f}]  x{t[a.reps // 2] / base:.3f}")

    # launches only the input-gradient variant issues, timed with CUDA events around each launch (profiled pass)
    ops.PROFILE_DETAIL = True
    prof = {}
    for name in ("fused, x without grad", "fused, x.requires_grad_()"):
        ops.profile_begin()
        variants[name]()
        prof[name] = ops.profile_end()
    ops.PROFILE_DETAIL = False
    plain, withg = prof["fused, x without grad"], prof["fused, x.requires_grad_()"]
    print("launches added by the input gradient (profiled pass, CUDA events around each launch):")
    extra_ms = 0.0
    for label, (ms, cnt) in sorted(withg.items()):
        ms0, cnt0 = plain.get(label, (0.0, 0))
        if cnt > cnt0:
            dms = ms - ms0
            extra_ms += dms
            print(f"  {label:90s} +{cnt - cnt0} launch(es) {dms:8.3f} ms")
    n, hw = a.batch, a.size
    p = 4
    nbytes = n * (hw + 2 * p) ** 2 * 3 * 4 + n * 3 * hw * hw * 4         # fp32 gpad read + fp32 NCHW gradient written
    fold = [(lbl, v) for lbl, v in withg.items() if "reflect_fold" in lbl]
    for lbl, (ms, cnt) in fold:
        print(f"  ast_reflect_fold: {ms / cnt:.4f} ms per launch, {nbytes / 1e6:.1f} MB moved, "
              f"{nbytes / (ms / cnt * 1e-3) / 1e9:.0f} GB/s achieved")
    print(f"  sum of the added launches: {extra_ms:.3f} ms")


if __name__ == "__main__":
    main()
