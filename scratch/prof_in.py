"""Micro-benchmark of the InstanceNorm kernels on the residual-block shape (B=32, 64x64x128 bf16) and the 256^2x32 shape.
Rotates over several buffer sets (> L2) so x is read from HBM like in the real step."""
import sys, torch
sys.path.insert(0, '.')
from artist_style_transfer_b200 import ops
torch.manual_seed(0)
def bench(n, h, w, c, pad, relu, residual, sets=6, iters=30):
    dt = torch.bfloat16
    bufs = []
    for _ in range(sets):
        x = torch.randn(n, h, w, c, device='cuda').to(dt)
        gp = torch.randn(n, h + 2 * pad, w + 2 * pad, c, device='cuda').to(dt)
        ge = torch.randn(n, h, w, c, device='cuda').to(dt) if residual else None
        dx = torch.empty_like(x)
        gt = torch.empty_like(x) if residual else None
        out = torch.empty(n, h + 2 * pad, w + 2 * pad, c, device='cuda', dtype=dt)
        bufs.append((x, gp, ge, dx, gt, out))
    mean = torch.randn(n * c, device='cuda'); rstd = torch.rand(n * c, device='cuda') + 0.5
    gam = torch.randn(c, device='cuda'); bet = torch.randn(c, device='cuda')
    s12 = torch.zeros(64, 2, n * c, device='cuda')
    arrive = torch.zeros(64, n, dtype=torch.int32, device='cuda')
    def run_bwd(i):                 # zeroed sums / counters: a fresh slice per call
        x, gp, ge, dx, gt, out = bufs[i % sets]
        ops._instnorm_bwd_impl(x, mean, rstd, gam, bet, gp, pad, ge, relu, dx, gtotal=gt, s12=s12[i % 64],
                               arrive=arrive[i % 64])
    def run_apply(i):
        x, gp, ge, dx, gt, out = bufs[i % sets]
        ops._instnorm_apply_impl(x, mean, rstd, gam, bet, out, pad, relu, residual=ge)
    for name, fn, nbytes in (("bwd", run_bwd, (x.numel() * (2 + 1 + (2 if residual else 0)) + gp.numel() * 2) * 2),
                             ("apply", run_apply, (x.numel() * (1 + (1 if residual else 0)) + out.numel()) * 2)):
        for i in range(5): fn(i)
        torch.cuda.synchronize()
        s12.zero_(); arrive.zero_()
        graph = torch.cuda.CUDAGraph()                 # graph replay: no CPU launch overhead in the timing
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            fn(0)
            with torch.cuda.graph(graph, stream=st):
                for i in range(iters): fn(i)
        torch.cuda.synchronize()
        graph.replay(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        print(f"{name:6s} ({n},{h},{w},{c}) pad={pad} res={residual}: {ms*1e3:7.1f} us  {nbytes/ms/1e6:7.0f} GB/s (all passes' bytes)")
bench(32, 64, 64, 128, 1, True, False)
bench(32, 64, 64, 128, 1, False, True)
bench(32, 256, 256, 32, 4, True, False, sets=3)
bench(32, 128, 128, 64, 1, True, False, sets=4)
