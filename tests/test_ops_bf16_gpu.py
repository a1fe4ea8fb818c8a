"""bf16 per-op pins (VERDICT r01 weak #1): the fast-mode backward kernels against torch fp64 evaluated on the SAME
bf16-rounded operands.  fp32 outputs are pinned at 1e-5; bf16 outputs element-wise to one bf16 rounding (2^-8 relative +
1e-5 of the tensor's scale), which is as tight as a bf16 store allows.  Production tile shapes (>= 64^2 images), and the
kernel family that ran is asserted through the library's per-family launch counters."""
import pytest
import torch
import torch.nn.functional as F

from test_instnorm_launch_kernels import check_bwd, probe_failures

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from artist_style_transfer_b200 import _lib, conv_geometry as cg, ops
    if not _lib.has_tc_conv():
        pytest.skip("library built without the tcgen05 kernels")
    return _lib, cg, ops


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def assert_bf16_close(got, ref, what=""):
    got, ref = got.double().cpu(), ref.double().cpu()
    tol = ref.abs() * 2.0 ** -8 + 1e-5 * float(ref.abs().max())
    bad = (got - ref).abs() > tol
    assert not bool(bad.any()), (what, int(bad.sum()), float(((got - ref).abs() / (tol + 1e-30)).max()))


def bf(x):
    return x.to(torch.bfloat16)


def instnorm_bwd_reference(x, gamma, beta, gpad, pad, gextra, relu):
    """fp64 backward of ReflectionPad o ReLU o (+residual) o InstanceNorm on the device (CPU autograd at 10^8 elements is
    too slow) -> fp32 mean / rstd, dbeta, dgamma, dx and g' (NHWC; g' only with gextra; gpad may be None)."""
    xd = x.double().permute(0, 3, 1, 2).requires_grad_(True)
    gd, bd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    y = F.instance_norm(xd, weight=gd, bias=bd, eps=1e-5)
    if relu:
        y = F.relu(y)
    yp = F.pad(y, (pad,) * 4, mode="reflect") if pad else y
    loss = (yp * gpad.double().permute(0, 3, 1, 2)).sum() if gpad is not None else 0
    if gextra is not None:
        loss = loss + (y * gextra.double().permute(0, 3, 1, 2)).sum()
    loss.backward()
    mean = xd.detach().mean(dim=(2, 3)).reshape(-1).float()
    rstd = (xd.detach().var(dim=(2, 3), unbiased=False) + 1e-5).rsqrt().reshape(-1).float()
    gprime = None
    if gextra is not None:
        yr = F.instance_norm(xd.detach(), weight=gd.detach(), bias=bd.detach(), eps=1e-5)
        fold = 0
        if gpad is not None:
            gp = gpad.double().permute(0, 3, 1, 2)
            fold = torch.autograd.functional.vjp(lambda t: F.pad(t, (pad,) * 4, mode="reflect") if pad else t, yr, gp)[1]
        gprime = ((fold + gextra.double().permute(0, 3, 1, 2)) * ((yr > 0) if relu else 1.0)).permute(0, 2, 3, 1)
    return mean, rstd, bd.grad, gd.grad, xd.grad.permute(0, 2, 3, 1), gprime


@pytest.mark.parametrize("dt,n,h,w,c,pad,relu,res,launches", [
    # x + g' small enough to stay in L2: one cooperative kernel
    ("bf16", 2, 64, 64, 128, 1, True, False, 1), ("bf16", 2, 64, 64, 128, 1, False, True, 1),
    ("bf16", 1, 128, 128, 64, 1, True, False, 1), ("bf16", 1, 96, 80, 32, 4, True, False, 1),
    ("bf16", 2, 64, 64, 128, 0, True, False, 1), ("fp32", 2, 64, 64, 128, 1, True, False, 1),
    # production layers too large for L2: statistics, then apply
    ("bf16", 32, 128, 128, 64, 1, True, False, 2), ("bf16", 32, 256, 256, 32, 4, True, False, 2),
    ("bf16", 16, 128, 128, 128, 1, False, True, 2), ("fp32", 32, 128, 128, 64, 1, True, False, 2),
    # the staging plan's edges: a row of 257 pixels in two segments; three staged tensors (8 KB slabs) of 70 pixels in
    # segments of 24, 24 and 22; pad 4 at h = w = 5 (every pixel folds mirrored positions)
    ("bf16", 2, 9, 257, 32, 1, True, False, 1), ("bf16", 2, 16, 70, 128, 1, False, True, 1),
    ("bf16", 2, 5, 5, 32, 4, True, False, 1), ("fp32", 2, 5, 5, 32, 4, False, True, 1),
    # the channel counts at both ends of the consumer mapping (1 lane x 256 slots .. 128 lanes x 2 slots)
    ("bf16", 2, 64, 64, 8, 1, True, False, 1), ("bf16", 2, 16, 16, 1024, 1, True, False, 1),
    ("fp32", 2, 32, 32, 4, 1, True, False, 1), ("fp32", 2, 16, 16, 512, 1, True, False, 1),
    # n = 1: one row per block; n = 300: one block per image, more blocks than fit at once -> two launches in L2
    ("bf16", 1, 64, 64, 32, 1, True, False, 1), ("bf16", 300, 8, 8, 32, 1, True, False, 2),
    # the L2 rule: x + g' of 103.7 MB and of 104.6 MB
    ("bf16", 4, 225, 225, 128, 1, True, False, 1), ("bf16", 4, 226, 226, 128, 1, True, False, 2),
    # only the skip gradient (no padded gradient)
    ("bf16", 2, 64, 64, 128, 1, True, "only", 1),
    # |mean| / std = 100 and 1000: sums of g' * xhat must stay within the conditioning of the maths (a sum of g' * x
    # corrected by mean * sum g' afterwards does not: 2.3e-5 off in dgamma at 100, fp32, two launches).  fp32 without
    # ReLU: at this ratio fp32 D = beta - A*mean moves the ReLU threshold by ~1e-5 std, which flips masks against the
    # exact-mask norm pins below (check_bwd evaluates the mask as the kernel does)
    ("bf16-mu100", 2, 64, 64, 128, 1, True, False, 1), ("fp32-mu100", 2, 64, 64, 128, 1, False, False, 1),
    ("fp32-mu100", 16, 128, 128, 64, 1, False, True, 2), ("fp32-mu1000", 2, 64, 64, 128, 1, False, True, 1)])
def test_instnorm_bwd_staged_bf16(env, dt, n, h, w, c, pad, relu, res, launches):
    """Backward of ReflectionPad o ReLU o (+residual) o InstanceNorm (cnn.py:58,68,91,98) against fp64 on the same rounded
    operands, on both sides of the library's size rule: the single cooperative kernel (second read from L2) and the
    two launches give the same numbers.  res: the skip gradient gextra (and gtotal); "only": gextra without gpad.  A
    "-muR" dtype draws x with |mean| / std = R.  Besides the norm-wise pins, every output is held element-wise to
    the bounds of `check_bwd` (test_instnorm_launch_kernels.py), whose sum bounds scale with sum |g' * xhat|."""
    _lib, cg, ops = env
    torch.manual_seed(c + h + pad)
    dt, _, mu = dt.partition("-")
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    x = ((torch.randn(n, h, w, c, device="cuda") * (2 / int(mu[2:])) + 2) if mu else
         (torch.randn(n, h, w, c, device="cuda") * 2 + 0.5)).to(dtype)
    gamma = torch.rand(c, device="cuda") + 0.5
    beta = torch.randn(c, device="cuda") * 0.3
    gpad = torch.randn(n, h + 2 * pad, w + 2 * pad, c, device="cuda").to(dtype) if res != "only" else None
    gextra = torch.randn(n, h, w, c, device="cuda").to(dtype) if res else None
    mean, rstd, dbeta, dgamma, dx_ref, gprime = instnorm_bwd_reference(x, gamma, beta, gpad, pad, gextra, relu)
    dx = torch.full_like(x, float("nan"))
    gtotal = torch.full_like(x, float("nan")) if res else None
    s12 = torch.zeros(2, n * c, device="cuda")
    arrive = torch.zeros(n, dtype=torch.int32, device="cuda")
    before = _lib.family_stats()
    ops.instnorm_bwd(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal, s12=s12, arrive=arrive)
    assert _lib.family_delta(before)["in_bwd"][0] == launches, f"{launches} InstanceNorm backward launch(es) expected"
    if launches == 1:
        assert int(arrive.min()) == int(arrive.max()) > 0
    rec = check_bwd(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal, s12,
                    torch.cuda.get_device_properties(0).multi_processor_count)
    print(f"{(dt, mu, n, h, w, c, pad, relu, res)}: plan {rec['plan']}, k {rec['k']}: max err/bound dx "
          f"{rec['ratio_dx']:.2e}, sums {rec['ratio_sums']:.2e}, all {rec['ratio']:.2e}; "
          f"dgamma rel {rel(s12[1].view(n, c).sum(0), dgamma):.1e}; mutants {rec['mutants']}")
    assert rec["plan"]["launches"] == launches
    rec.update(entry="bwd", fams={}, want={}, inputs_changed=[], zero_on_entry=True,
               arrive=(int(arrive.min()), int(arrive.max())))
    assert not probe_failures(rec), probe_failures(rec)
    if mu != "mu1000":   # there the fp32 rounding of the mean alone moves xhat by 6e-5 std against exact statistics
        assert rel(s12[0].view(n, c).sum(0), dbeta) < 1e-5          # dbeta = sum g'
        assert rel(s12[1].view(n, c).sum(0), dgamma) < 2e-5         # dgamma = sum g' xhat
    assert_bf16_close(dx, dx_ref, "dx")
    if res:        # gtotal = g' (the gradient handed to the residual skip)
        assert_bf16_close(gtotal, gprime, "gtotal")


def test_instnorm_images_more_than_2g_elements_apart(env):
    """Strict-mode batches can span more than 2^31 elements: the staged InstanceNorm kernels address image and row starts
    in 64 bits.  Two images 2^31 + 1024 elements apart (views into one 4.3 GB buffer): the apply output is bit-identical
    to the one computed from compact copies, and the backward meets the fp64 bounds of the test above."""
    _lib, cg, ops = env
    torch.manual_seed(7)
    n, h, w, c, pad = 2, 64, 64, 128, 1
    hp, wp = h + 2 * pad, w + 2 * pad
    sn = 2 ** 31 + 1024
    big = torch.empty(sn + 4 * h * w * c + 2 * hp * wp * c, dtype=torch.bfloat16, device="cuda")
    off = 0

    def view(hh, ww):        # per image: x | residual | dx | gtotal | gpad | out, the images sn elements apart
        nonlocal off
        v = big.as_strided((n, hh, ww, c), (sn, ww * c, c, 1), off)
        off += hh * ww * c
        return v
    x, res, dx, gtotal, gpad, out = view(h, w), view(h, w), view(h, w), view(h, w), view(hp, wp), view(hp, wp)
    for t in (x, res, gpad):
        t.copy_(torch.randn(t.shape, device="cuda"))
    gamma = torch.rand(c, device="cuda") + 0.5
    beta = torch.randn(c, device="cuda") * 0.3
    mean, rstd, dbeta, dgamma, dx_ref, gprime = instnorm_bwd_reference(x, gamma, beta, gpad, pad, res, True)

    ops.instnorm_apply(x, mean, rstd, gamma, beta, out, pad, True, residual=res)
    out_c = torch.empty(out.shape, dtype=out.dtype, device="cuda")
    ops.instnorm_apply(x.contiguous(), mean, rstd, gamma, beta, out_c, pad, True, residual=res.contiguous())
    assert torch.equal(out, out_c)

    s12 = ops.instnorm_bwd(x, mean, rstd, gamma, beta, gpad, pad, res, True, dx, gtotal)
    assert rel(s12[0].view(n, c).sum(0), dbeta) < 1e-5
    assert rel(s12[1].view(n, c).sum(0), dgamma) < 2e-5
    assert_bf16_close(dx, dx_ref, "dx")
    assert_bf16_close(gtotal, gprime, "gtotal")


def test_maxpool2_bwd_and_mask_add_bf16(env):
    """gx = (route(gy) + gadd) * (x > 0) (VGG pool backward fused with the tap-gradient add and ReLU mask) and
    out = (a + b) * (mask > 0), bf16 gradients, fp32 features."""
    _lib, cg, ops = env
    torch.manual_seed(3)
    n, h, w, c = 2, 64, 64, 128
    x = torch.relu(torch.randn(n, h, w, c, device="cuda"))
    gy = bf(torch.randn(n, h // 2, w // 2, c, device="cuda"))
    gadd = torch.randn(n, h, w, c, device="cuda")
    gx = ops.maxpool2_bwd(x, gy, gadd)
    xd = x.double().cpu().permute(0, 3, 1, 2)
    pooled, idx = F.max_pool2d(xd, 2, 2, return_indices=True)
    route = F.max_unpool2d(gy.double().cpu().permute(0, 3, 1, 2), idx, 2, 2, output_size=xd.shape[-2:])
    ref = ((route + gadd.double().cpu().permute(0, 3, 1, 2)) * (xd > 0)).permute(0, 2, 3, 1)
    assert gx.dtype == torch.bfloat16
    assert_bf16_close(gx, ref, "maxpool2_bwd")
    a, b = torch.randn(n, 32, 32, 512, device="cuda"), bf(torch.randn(n, 32, 32, 512, device="cuda"))
    mask = torch.relu(torch.randn(n, 32, 32, 512, device="cuda"))
    out = torch.empty(a.shape, dtype=torch.bfloat16, device="cuda")
    ops.mask_add(a, b, mask, out)
    assert_bf16_close(out, (a.double() + b.double()) * (mask > 0), "mask_add")


def test_pool_window_codes(env):
    """The 1-byte window codes (arg max + four ReLU bits) written by ast_maxpool2_fwd and by the fused conv1_2 + pool
    epilogue let ast_maxpool2_bwd run without the activations: identical results to the path that re-reads x."""
    _lib, cg, ops = env
    torch.manual_seed(5)
    n, h, w, c = 2, 64, 48, 128
    x = torch.relu(torch.randn(n, h, w, c, device="cuda"))
    x[0, :2, :2, :] = 0.0                                       # ties (all-zero windows): first maximum wins, mask off
    gy = bf(torch.randn(n, h // 2, w // 2, c, device="cuda"))
    gadd = bf(torch.randn(n, h, w, c, device="cuda"))
    codes = torch.empty(n, h // 2, w // 2, c, dtype=torch.uint8, device="cuda")
    y = ops.maxpool2_fwd(x, codes=codes)
    assert torch.equal(y, F.max_pool2d(x.permute(0, 3, 1, 2), 2, 2).permute(0, 2, 3, 1))
    ref = ops.maxpool2_bwd(x, gy, gadd)
    got = ops.maxpool2_bwd(None, gy, gadd, codes=codes)
    assert torch.equal(ref, got)
    assert torch.equal(ops.maxpool2_bwd(x, gy, None), ops.maxpool2_bwd(None, gy, None, codes=codes))
    # the fused conv + ReLU + pool epilogue writes the same codes as the stand-alone pooling kernel on its own output
    xin = torch.randn(n, 32, 40, 64, device="cuda").half()        # fp16 activations in, fp32 tap + fp16 pooled tensor out
    wt = torch.randn(64, 64, 3, 3, device="cuda") / 24
    launches = cg.conv_fwd(3, 1, 1, 32, 40)
    wp = ops.pack_weights(wt, launches, 64, 64, 64 * 9, 9, 3, 1, torch.float32).half()
    full = torch.empty(n, 32, 40, 64, device="cuda")
    pooled = torch.empty(n, 16, 20, 64, device="cuda", dtype=torch.float16)
    fcodes = torch.empty(n, 16, 20, 64, dtype=torch.uint8, device="cuda")
    ops.conv_gather(xin, wp, launches, full, relu=True, tensor=True, round_tf32=True, pooled=pooled, pool_codes=fcodes)
    codes2 = torch.empty_like(fcodes)
    pooled2 = ops.maxpool2_fwd(full, codes=codes2, out_dtype=torch.float16)
    assert torch.equal(pooled, pooled2) and torch.equal(fcodes, codes2)


@pytest.mark.parametrize("cin,cout,size,family", [(128, 128, 128, "conv_hx"), (64, 64, 256, "conv_ws"),
                                                   (256, 128, 64, "conv_hx"), (512, 512, 32, "conv_hx"),
                                                   (128, 64, 128, "conv_ws"), (512, 256, 33, "conv_hx")])
def test_vgg_dgrad_with_add_and_mask_production_tiles(env, cin, cout, size, family):
    """Data gradient of a VGG 3x3 conv (train_cnn.py:54) with the tap-gradient add and the ReLU mask in the epilogue, bf16
    gradients, at the image sizes of the B=32 step: conv_hx (halo kernel, cout % 128 == 0), conv_ws (conv1_2's 64->64 at
    256^2), conv_px (cout 64 with a filter too large for conv_ws); one ragged size (33) for the tile-edge predicates."""
    _lib, cg, ops = env
    torch.manual_seed(cin + size)
    n = 1
    g = bf(torch.randn(n, size, size, cin, device="cuda"))               # gradient w.r.t. the conv OUTPUT (cin = its cout)
    wt = torch.randn(cin, cout, 3, 3, device="cuda") / (cin * 9) ** 0.5  # conv weight (Co=cin here, Ci=cout)
    launches = cg.conv_dgrad(3, 1, 1, size, size)
    wp = ops.pack_weights(wt, launches, cout, cin, 9, cout * 9, 3, 1, torch.bfloat16)    # [t][ci][co]
    add = torch.randn(n, size, size, cout, device="cuda")
    mask = torch.relu(torch.randn(n, size, size, cout, device="cuda"))
    out = torch.full((n, size, size, cout), float("nan"), dtype=torch.bfloat16, device="cuda")
    before = _lib.family_stats()
    ops.conv_gather(g, wp, launches, out, add=add, mask=mask, tensor=True)
    delta = _lib.family_delta(before)
    assert delta[family][0] == 1, {k: v[0] for k, v in delta.items() if v[0]}
    ref = F.conv_transpose2d(g.double().cpu().permute(0, 3, 1, 2), bf(wt).double().cpu(), padding=1).permute(0, 2, 3, 1)
    ref = (ref + add.double().cpu()) * (mask.double().cpu() > 0)
    assert_bf16_close(out, ref, family)


@pytest.mark.parametrize("cin,cout,size,family", [(64, 128, 130, "conv_px"), (32, 64, 258, "conv_px"), (128, 128, 66, "conv_hx")])
def test_transform_convs_with_fused_statistics(env, cin, cout, size, family):
    """Forward convs of the TransformerNet on physically padded bf16 inputs (cnn.py:18-20 stride 2, :26-30 residual) with
    the InstanceNorm sums accumulated by the epilogue: raw output to one bf16 rounding, mean / rstd against fp64."""
    _lib, cg, ops = env
    torch.manual_seed(cin + size)
    n = 2
    stride = 2 if family != "conv_hx" else 1
    x = bf(torch.randn(n, size, size, cin, device="cuda"))
    wt = torch.randn(cout, cin, 3, 3, device="cuda") / (cin * 9) ** 0.5
    launches = cg.conv_fwd(3, stride, 0, size, size)
    ho = launches[0].mi
    wp = ops.pack_weights(wt, launches, cout, cin, cin * 9, 9, 3, 1, torch.bfloat16)
    raw = torch.full((n, ho, ho, cout), float("nan"), dtype=torch.bfloat16, device="cuda")
    sums = torch.zeros(2 * n * cout, dtype=torch.float64, device="cuda")
    before = _lib.family_stats()
    ops.conv_gather(x, wp, launches, raw, tensor=True, stats=sums)
    delta = _lib.family_delta(before)
    assert delta[family][0] == 1, {k: v[0] for k, v in delta.items() if v[0]}
    mean, rstd = ops.instnorm_finalize(sums, n, cout, ho * ho)
    y = F.conv2d(x.double().cpu().permute(0, 3, 1, 2), bf(wt).double().cpu(), stride=stride)
    assert_bf16_close(raw, y.permute(0, 2, 3, 1), family)
    assert rel(mean, y.mean(dim=(2, 3)).reshape(-1)) < 1e-4
    assert rel(rstd, (y.var(dim=(2, 3), unbiased=False) + 1e-5).rsqrt().reshape(-1)) < 1e-5


def test_fused_instnorm_statistics_survive_large_mean(env):
    """A conv output plane with |mean| / std = 100 (SURVEY section 7: E[x^2] - mean^2 cancels in fp32): the statistics fused
    into the tcgen05 epilogues are accumulated in fp64 from centred / short fp32 partial sums, so mean and rstd still
    match fp64 statistics of the same conv output."""
    _lib, cg, ops = env
    torch.manual_seed(0)
    for cin, cout, size in [(128, 128, 64), (32, 64, 64), (64, 32, 128)]:
        n = 2
        x = bf(torch.randn(n, size + 2, size + 2, cin, device="cuda") * 0.5 + 3.0)
        wt = 0.03 * torch.randn(cout, cin, 3, 3, device="cuda") / (cin * 9) ** 0.5
        wt = wt - wt.mean(dim=(1, 2, 3), keepdim=True) + 0.55 / (cin * 9)        # output mean ~ 3 * 0.55, std ~ 0.015
        launches = cg.conv_fwd(3, 1, 0, size + 2, size + 2)
        wp = ops.pack_weights(wt, launches, cout, cin, cin * 9, 9, 3, 1, torch.bfloat16)
        raw = torch.empty((n, size, size, cout), dtype=torch.bfloat16, device="cuda")
        sums = torch.zeros(2 * n * cout, dtype=torch.float64, device="cuda")
        ops.conv_gather(x, wp, launches, raw, tensor=True, stats=sums)
        mean, rstd = ops.instnorm_finalize(sums, n, cout, size * size)
        y = F.conv2d(x.double().cpu().permute(0, 3, 1, 2), bf(wt).double().cpu())
        m_ref = y.mean(dim=(2, 3)).reshape(-1)
        v_ref = y.var(dim=(2, 3), unbiased=False).reshape(-1)
        ratio = float((m_ref.abs() / v_ref.sqrt()).median())
        assert ratio > 50, ratio
        assert rel(mean, m_ref) < 5e-6          # fp32 accumulation of the 9*cin-term conv sums
        r_ref = (v_ref + 1e-5).rsqrt()
        assert float(((rstd.double().cpu() - r_ref).abs() / r_ref).max()) < 2e-3, (cin, cout)
