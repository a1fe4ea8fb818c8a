"""Per-layer parity (forward AND parameter gradients) of the CUDA kernels against torch.nn.functional in fp64
on CPU - the op-level tier of SURVEY.md section 4.  Tolerances: strict fp32 mode 1e-5-class; bf16 mode as stated."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def ast():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import artist_style_transfer_b200 as m
    return m


def _ref_conv_layer(x, w, b, g, be, k, s, norm=True):
    xp = F.pad(x, (k // 2,) * 4, mode="reflect") if k > 1 else x
    y = F.conv2d(xp, w, b, stride=s)
    return F.instance_norm(y, weight=g, bias=be, eps=1e-5) if norm else y


@pytest.mark.parametrize("cin,cout,k,s,h,w,norm", [
    (3, 32, 9, 1, 24, 28, "instance"), (32, 64, 3, 2, 20, 24, "instance"), (64, 128, 3, 2, 16, 16, "instance"),
    (128, 128, 1, 1, 9, 7, "instance"), (32, 3, 9, 1, 20, 20, "None"), (128, 128, 3, 1, 10, 12, "instance")])
def test_conv_layer_fp32(ast, cin, cout, k, s, h, w, norm):
    torch.manual_seed(cin + cout + k)
    layer = ast.ConvLayer(cin, cout, k, s, norm=norm).cuda()
    layer.precision = "fp32"
    if norm == "instance":
        with torch.no_grad():
            layer.norm_layer.weight.add_(0.3 * torch.randn(cout, device="cuda"))
            layer.norm_layer.bias.add_(0.3 * torch.randn(cout, device="cuda"))
    x = (torch.randn(2, cin, h, w) * 50).cuda()
    y = layer(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    P = {n: p.detach().double().cpu().requires_grad_(True) for n, p in layer.named_parameters()}
    yr = _ref_conv_layer(x.double().cpu(), P["conv_layer.weight"], P["conv_layer.bias"],
                         P.get("norm_layer.weight"), P.get("norm_layer.bias"), k, s, norm == "instance")
    yr.backward(gy.double().cpu())
    assert rel(y, yr) < 2e-6
    for n, p in layer.named_parameters():
        if n == "conv_layer.bias" and norm == "instance":
            assert float(p.grad.abs().max()) == 0.0            # dead parameter under InstanceNorm
            continue
        assert rel(p.grad, P[n].grad) < 2e-5, n


@pytest.mark.parametrize("cin,cout,k,s,op,h,w", [(128, 128, 1, 1, 0, 8, 8), (128, 64, 3, 2, 1, 8, 10), (64, 32, 3, 2, 1, 9, 8)])
def test_deconv_layer_fp32(ast, cin, cout, k, s, op, h, w):
    torch.manual_seed(5)
    layer = ast.DeconvLayer(cin, cout, k, s, op).cuda()
    layer.precision = "fp32"
    x = torch.randn(2, cin, h, w).cuda()
    y = layer(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    P = {n: p.detach().double().cpu().requires_grad_(True) for n, p in layer.named_parameters()}
    yr = F.conv_transpose2d(x.double().cpu(), P["conv_transpose.weight"], P["conv_transpose.bias"], stride=s,
                            padding=k // 2, output_padding=op)
    yr = F.instance_norm(yr, weight=P["norm_layer.weight"], bias=P["norm_layer.bias"], eps=1e-5)
    yr.backward(gy.double().cpu())
    assert rel(y, yr) < 2e-6
    for n in ("conv_transpose.weight", "norm_layer.weight", "norm_layer.bias"):
        assert rel(dict(layer.named_parameters())[n].grad, P[n].grad) < 2e-5, n


def test_residual_layer_fp32(ast):
    torch.manual_seed(7)
    layer = ast.ResidualLayer(128, 3).cuda()
    layer.precision = "fp32"
    x = torch.randn(2, 128, 12, 10).cuda()
    y = layer(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    P = {n: p.detach().double().cpu().requires_grad_(True) for n, p in layer.named_parameters()}
    xr = x.double().cpu()
    t = F.relu(_ref_conv_layer(xr, P["conv1.conv_layer.weight"], P["conv1.conv_layer.bias"],
                               P["conv1.norm_layer.weight"], P["conv1.norm_layer.bias"], 3, 1))
    yr = _ref_conv_layer(t, P["conv2.conv_layer.weight"], P["conv2.conv_layer.bias"],
                         P["conv2.norm_layer.weight"], P["conv2.norm_layer.bias"], 3, 1) + xr
    yr.backward(gy.double().cpu())
    assert rel(y, yr) < 2e-6
    for n, p in layer.named_parameters():
        if n.endswith("conv_layer.bias"):
            continue
        assert rel(p.grad, P[n].grad) < 3e-5, n


def test_conv_layer_bf16(ast):
    """bf16 activations/weights, fp32 accumulate: ~3 significant digits."""
    torch.manual_seed(11)
    layer = ast.ConvLayer(128, 128, 3, 1).cuda()
    layer.precision = "fast"
    x = torch.randn(2, 128, 16, 16).cuda()
    y = layer(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    P = {n: p.detach().double().cpu().requires_grad_(True) for n, p in layer.named_parameters()}
    yr = _ref_conv_layer(x.double().cpu(), P["conv_layer.weight"], P["conv_layer.bias"],
                         P["norm_layer.weight"], P["norm_layer.bias"], 3, 1)
    yr.backward(gy.double().cpu())
    assert rel(y, yr) < 1e-2
    assert rel(layer.conv_layer.weight.grad, P["conv_layer.weight"].grad) < 3e-2


def test_gram_and_mse(ast):
    from oracle import port
    torch.manual_seed(3)
    f = torch.randn(3, 64, 20, 12, device="cuda", requires_grad=True)
    target = torch.randn(3, 64, 64, device="cuda") * 0.1
    g = ast.gram(f, precision="fp32")
    loss = torch.nn.functional.mse_loss(g, target)          # the reference call site: nn.MSELoss on gram()
    loss.backward()
    fr = f.detach().double().cpu().requires_grad_(True)
    gr = port.gram(fr)
    lr = torch.nn.functional.mse_loss(gr, target.double().cpu())
    lr.backward()
    assert rel(g, gr) < 1e-6
    assert rel(f.grad, fr.grad) < 1e-5
    assert float((g - g.transpose(1, 2)).abs().max()) < 1e-6
    # fused MSE
    a = torch.randn(2, 8, 6, 6, device="cuda", requires_grad=True)
    b = torch.randn(2, 8, 6, 6, device="cuda")
    l2 = ast.mse_loss(a, b) * 17
    l2.backward()
    ar = a.detach().double().cpu().requires_grad_(True)
    lr2 = torch.nn.functional.mse_loss(ar, b.double().cpu()) * 17
    lr2.backward()
    assert abs(float(l2) - float(lr2)) < 1e-5 * abs(float(lr2))
    assert rel(a.grad, ar.grad) < 1e-6


@pytest.mark.parametrize("shape", [(0, 64, 8, 8), (1, 64, 1, 1), (2, 512, 3, 5)])
def test_gram_edge_shapes(ast, shape):
    from oracle import port
    f = torch.randn(shape, device="cuda")
    g = ast.gram(f, precision="fp32")
    assert g.shape == (shape[0], shape[1], shape[1])
    if shape[0]:
        assert rel(g, port.gram(f.double().cpu())) < 1e-6


@pytest.mark.parametrize("cin,cout,k,norm,h,w", [(3, 32, 9, "instance", 24, 28), (32, 3, 9, "None", 20, 24)])
def test_thin_layers_fast_mode(ast, cin, cout, k, norm, h, w):
    """The 3-channel 9x9 ends in bf16 on the tcgen05 kernels (row-im2col path) against torch fp64."""
    torch.manual_seed(21)
    layer = ast.ConvLayer(cin, cout, k, 1, norm=norm).cuda()
    layer.precision = "fast"
    x = torch.randint(0, 256, (2, cin, h, w)).float().cuda() if cin == 3 else torch.randn(2, cin, h, w).cuda()
    y = layer(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    P = {n: p.detach().double().cpu().requires_grad_(True) for n, p in layer.named_parameters()}
    yr = _ref_conv_layer(x.double().cpu(), P["conv_layer.weight"], P["conv_layer.bias"],
                         P.get("norm_layer.weight"), P.get("norm_layer.bias"), k, 1, norm == "instance")
    yr.backward(gy.double().cpu())
    assert rel(y, yr) < 1e-2
    assert rel(layer.conv_layer.weight.grad, P["conv_layer.weight"].grad) < 2e-2
    if norm == "None":
        assert rel(layer.conv_layer.bias.grad, P["conv_layer.bias"].grad) < 1e-4


@pytest.mark.parametrize("w", [13, 300])          # 300: wider than one 256-column block segment
def test_fold_rows_matches_direct_sum(ast, w):
    """ast_fold_rows: out[n,y,x,c] = bias[c] + sum_d part[n,y,x+d,d*C+c] (NCHW output view, optional ReLU)."""
    from artist_style_transfer_b200 import ops
    torch.manual_seed(5)
    n, h, c, k = 2, 7, 3, 9
    part = torch.randn(n, h, w + k - 1, 32, device="cuda")
    bias = torch.randn(c, device="cuda")
    out = torch.empty(n, c, h, w, device="cuda")
    ops.fold_rows(part, out.permute(0, 2, 3, 1), k, bias=bias, relu=False)
    ref = bias.view(1, 1, 1, c).expand(n, h, w, c).clone()
    for d in range(k):
        ref += part[:, :, d:d + w, d * c:(d + 1) * c]
    assert torch.allclose(out.permute(0, 2, 3, 1), ref, rtol=1e-6, atol=1e-6)
    out2 = torch.empty(n, h, w, c, device="cuda", dtype=torch.bfloat16)
    ops.fold_rows(part, out2, k, relu=True)
    ref2 = torch.relu(ref - bias.view(1, 1, 1, c)).bfloat16()
    assert torch.allclose(out2.float(), ref2.float(), rtol=1e-2, atol=1e-2)
