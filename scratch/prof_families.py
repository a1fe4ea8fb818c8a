"""One representative launch of every kernel family at the shapes of the B=32, 256^2 step, bracketed by
cudaProfilerStart/Stop so that `ncu --profile-from-start off --set full` captures exactly these launches.
Prints the launch order (the ncu report lists kernels in the same order)."""
import sys, torch
sys.path.insert(0, '.')
import artist_style_transfer_b200 as ast
from artist_style_transfer_b200 import _lib, ops, conv_geometry as cg
torch.manual_seed(0)
dev = torch.device('cuda')
n = 32
bf, f32, f16 = torch.bfloat16, torch.float32, torch.float16
todo = []

def conv(name, dtype, cin, cout, hin, launches, hout, stats=False, mask=False, pooled=False, w_img=False, relu=False, odt=None,
         mask_dtype=f32):
    odt = odt or dtype
    x = torch.randn(n, hin, hin, cin, device=dev).to(dtype)
    y = torch.empty(n, hout, hout, cout, device=dev, dtype=odt)
    nt = sum(len(l.taps) for l in launches)
    if w_img:
        wp = (torch.randn(n, nt, cout, cin, device=dev) / cin ** 0.5).to(dtype)
    else:
        wp = (torch.randn(nt, cout, cin, device=dev) / (cin * nt) ** 0.5).to(dtype)
    sums = torch.zeros(2 * n * cout, dtype=torch.float64, device=dev) if stats else None
    m = torch.randn(n, hout, hout, cout, device=dev).to(mask_dtype) if mask else None
    pool = torch.empty(n, hout // 2, hout // 2, cout, device=dev, dtype=dtype) if pooled else None   # fp16 in production
    pcodes = torch.empty(n, hout // 2, hout // 2, cout, device=dev, dtype=torch.uint8) if pooled else None
    todo.append((name, lambda: ops.conv_gather(x, wp, launches, y, tensor=True, stats=sums, mask=m, pooled=pool, pool_codes=pcodes, relu=relu,
                                               w_img_stride=cout * cin * nt if w_img else 0, round_tf32=odt == f32 and dtype != bf)))

vt9 = [cg.Launch(256, 256, 1, 1, 0, 0, [(d, 0) for d in range(9)], [(d, 0) for d in range(9)], 0)]
conv("conv_ws fp16 VGG conv1_2 64->64 256^2 (fp32 tap out) +ReLU +fused MaxPool (fp16) +window codes", f16, 64, 64, 256, cg.conv_fwd(3, 1, 1, 256, 256), 256, pooled=True, relu=True, odt=f32)
conv("conv_ws bf16 VGG dgrad conv1_2 64->64 256^2 +fp16 mask", bf, 64, 64, 256, cg.conv_dgrad(3, 1, 1, 256, 256), 256, mask=True, mask_dtype=f16)

def stacked(name, dtype, odt, cin, cout, hw_in, hw_out, launches, stats=False, relu=False):
    from artist_style_transfer_b200 import arena as arena_mod
    x = torch.randn(n, hw_in[0], hw_in[1], cin, device=dev).to(dtype)
    y = torch.empty(n, hw_out[0], hw_out[1], cout, device=dev, dtype=odt)
    nt = sum(len(l.taps) for l in launches)
    wp = (torch.randn(nt, cout, cin, device=dev) / (cin * nt) ** 0.5).to(dtype)
    tidx = {wt: l.woff + t for l in launches for t, wt in enumerate(l.wtaps)}
    groups = arena_mod.stack_groups(launches, cout)
    ws = [ops.stack_filter(lambda pos: wp[tidx[pos]], g, cout, cin, dtype, dev) for g in groups]
    sums = torch.zeros(2 * n * cout, dtype=torch.float64, device=dev) if stats else None
    def go():
        for g, w in zip(groups, ws):
            ops.conv_stacked(x, w, g, y, stats=sums, relu=relu, round_tf32=dtype == f32)
    todo.append((name, go))

stacked("conv_st bf16 T first layer (9 vertical taps over row-im2col, 4 interleaved rows) 32->32 256^2 +stats", bf, bf, 32, 32, (264, 256), (256, 256), vt9, stats=True)
stacked("conv_st bf16 T ConvTranspose 3x3 s2 64->32 128^2->256^2 (4 phases stacked) +stats", bf, bf, 64, 32, (128, 128), (256, 256), cg.convT_fwd(3, 2, 1, 1, 128, 128), stats=True)
stacked("conv_st fp16 VGG conv1_1 (3 vertical taps, 2 interleaved rows) 32->64 256^2 +ReLU", f16, f16, 32, 64, (256, 256), (256, 256),
        [cg.Launch(256, 256, 1, 1, 0, 0, [(-1, 0), (0, 0), (1, 0)], [(0, 0), (1, 0), (2, 0)], 0)], relu=True)
conv("conv_hx bf16 T residual 3x3 128->128 64^2 +stats", bf, 128, 128, 66, cg.conv_fwd(3, 1, 0, 66, 66), 64, stats=True)
conv("conv_hx fp16 VGG conv2_2 128->128 128^2 (fp32 tap out)", f16, 128, 128, 128, cg.conv_fwd(3, 1, 1, 128, 128), 128, relu=True, odt=f32)
conv("conv_hx fp16 VGG conv4_2 512->512 32^2", f16, 512, 512, 32, cg.conv_fwd(3, 1, 1, 32, 32), 32, relu=True)
conv("conv_hx bf16 VGG dgrad conv3_2 256->256 64^2 +fp16 mask", bf, 256, 256, 64, cg.conv_dgrad(3, 1, 1, 64, 64), 64, mask=True, mask_dtype=f16)
conv("conv_px bf16 T conv 3x3 stride 2 64->128 130^2->64^2 +stats", bf, 64, 128, 130, cg.conv_fwd(3, 2, 0, 130, 130), 64, stats=True)
conv("conv_tc tf32 Gram backward relu2_2 (1x1, per-image weights) 128->128 128^2", f32, 128, 128, 128, cg.conv_fwd(1, 1, 0, 128, 128), 128, w_img=True)

# filter gradients
xw = torch.randn(n, 66, 66, 128, device=dev).to(bf); gw = torch.randn(n, 64, 64, 128, device=dev).to(bf)
dw = torch.zeros(3, 3, 128, 128, device=dev)
lw = cg.conv_fwd(3, 1, 0, 66, 66)
todo.append(("contract_tc bf16 wgrad residual 3x3 128x128", lambda: ops.wgrad_gather(xw, gw, lw, dw, 128, 1, 3 * 128 * 128, 128 * 128, tensor=True)))
xt = torch.randn(n, 264, 256, 32, device=dev).to(bf); gt = torch.randn(n, 256, 256, 32, device=dev).to(bf)
dwt = torch.zeros(9, 32, 32, device=dev)
todo.append(("contract_thin bf16 wgrad first layer (9 vertical taps)", lambda: ops.wgrad_gather(xt, gt, vt9, dwt, 32, 1, 32 * 32, 0, tensor=True)))
# Gram + fused style MSE
for c, s in ((64, 256), (512, 32)):
    f = torch.randn(n, s, s, c, device=dev); tgt = torch.randn(c, c, device=dev)
    g = torch.zeros(n, c, c, device=dev); cnt = torch.zeros(n * 16, dtype=torch.int32, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev); d = torch.empty(n, c, c, device=dev)
    def gm(f=f, tgt=tgt, g=g, cnt=cnt, loss=loss, d=d):
        g.zero_(); cnt.zero_()
        ops.gram_mse(f, tgt, g, cnt, loss=loss, loss_scale=1.0, d=d, d_scale=1.0, tensor=True)
    todo.append((f"contract_tc tf32 Gram + style MSE C={c} HW={s}^2", gm))
# InstanceNorm
xn = torch.randn(n, 64, 64, 128, device=dev).to(bf); gp = torch.randn(n, 66, 66, 128, device=dev).to(bf)
mean = torch.randn(n * 128, device=dev); rstd = torch.rand(n * 128, device=dev) + 0.5
gam = torch.randn(128, device=dev); bet = torch.randn(128, device=dev)
outp = torch.empty(n, 66, 66, 128, device=dev, dtype=bf); dxn = torch.empty_like(xn)
todo.append(("in_apply_staged bf16 64^2x128 +ReLU +reflect pad 1", lambda: ops.instnorm_apply(xn, mean, rstd, gam, bet, outp, 1, True)))
s12 = torch.zeros(2, n * 128, device=dev); arr = torch.zeros(n, dtype=torch.int32, device=dev)
def inb():
    s12.zero_(); arr.zero_()
    ops.instnorm_bwd(xn, mean, rstd, gam, bet, gp, 1, None, True, dxn, None, s12=s12, arrive=arr)
todo.append(("in_bwd_staged bf16 64^2x128 (stats + apply, one cooperative kernel)", inb))
xb = torch.randn(n, 256, 256, 32, device=dev).to(bf); gpb = torch.randn(n, 264, 264, 32, device=dev).to(bf)
mb = torch.randn(n * 32, device=dev); rb = torch.rand(n * 32, device=dev) + 0.5
dxb = torch.empty_like(xb)
todo.append(("in_bwd_staged bf16 256^2x32 pad 4 (stats, then apply: two launches)", lambda: ops.instnorm_bwd(xb, mb, rb, gam[:32].contiguous(), bet[:32].contiguous(), gpb, 4, None, True, dxb, None)))
# pointwise
xp = torch.relu(torch.randn(n, 256, 256, 64, device=dev)); gy = torch.randn(n, 128, 128, 64, device=dev).to(bf)
ga = torch.randn(n, 256, 256, 64, device=dev).to(bf)
codes = torch.empty(n, 128, 128, 64, dtype=torch.uint8, device=dev)
ops.maxpool2_fwd(xp, codes=codes)
todo.append(("maxpool2_bwd_codes 256^2x64 (1-byte window codes, bf16 gy, bf16 tap gradient)", lambda: ops.maxpool2_bwd(None, gy, ga, codes=codes)))
a2 = torch.randn(n, 128, 128, 128, device=dev); b2 = torch.randn(n, 128, 128, 128, device=dev)
l2 = torch.zeros(1, device=dev); gr = torch.empty_like(a2)
todo.append(("mse_vec 128^2x128 (content loss + gradient)", lambda: ops.mse(a2, b2, l2, 1.0, gr, 1.0)))
img = torch.randint(0, 256, (n, 3, 256, 256), device=dev, dtype=torch.uint8)
rim = torch.empty(n, 264, 256, 32, device=dev, dtype=bf)
todo.append(("row_im2col uint8 NCHW -> bf16 [n,264,256,32]", lambda: ops.row_im2col(img.permute(0, 2, 3, 1), rim, 9, 1, 4, 4, True)))
part = torch.randn(n, 256, 264, 32, device=dev); fo = torch.empty(n, 3, 256, 256, device=dev)
todo.append(("fold_rows [n,256,264,32] -> NCHW fp32", lambda: ops.fold_rows(part, fo.permute(0, 2, 3, 1), 9, bias=bet[:3].contiguous())))
# optimizer
net = ast.StyleTransfer(device=dev, precision='fast')
arena = net._arena_for(dev)
arena.enable_optimizer(2.4e-3)
gbuf = arena.new_grad_buffer().normal_()
todo.append(("adam_pack_kernel (Adam + L2 + bf16 re-pack of all 70 tensors)", lambda: arena.adam_step(gbuf)))

for _, fn in todo:      # warm-up (tensor maps, attributes)
    fn(); fn()
torch.cuda.synchronize()
torch.cuda.profiler.start()
for name, fn in todo:
    before = _lib.launch_count()
    fn()
    print(f"{_lib.launch_count() - before} launch(es): {name}")
torch.cuda.synchronize()
torch.cuda.profiler.stop()
