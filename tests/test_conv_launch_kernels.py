"""Every convolution launch of a training step, against fp64 of its own operands.

Every activation and every data gradient of a step comes out of `ops.conv_gather` (`ast_conv_gather`: conv_hx / conv_ws /
conv_px / conv_tc on the tensor cores in fast mode, conv_simt in strict mode) or `ops.conv_stacked` (`ast_conv_stacked`:
conv_st, or conv_hx when the stacked filter does not fit in shared memory); `ops.row_im2col` and `ops.fold_rows` complete
the 3-channel ends.  The step-level parity tests go through the whole network and must be loose; a launch wrong at one
halo edge, one partial tile or one cin chunk passes them.  Here a real `perceptual_step` runs with those four entry points
wrapped.  Each call fills the positions it is expected to write with NaN, runs once with unchanged arguments, and is
compared with an fp64 evaluation of exactly the operands it received, so the bounds are those of ONE fp32-accumulated
contraction.  Each call must also fill every position it owns, leave every other byte of its output's storage, its
inputs and its side outputs (fused statistics, pooled tensor, window codes) alone, and run the kernel family and launch
count that the dispatch promises.  For every call the test shows that the element-wise bound would catch the loss of one
tap on the last grid row of the last image (a halo or edge-tile bug), and, where they apply, a wrong image's weights, a
missing add and a missing mask.

The fp64 references are themselves checked against torch on the CPU."""
import inspect
import os
import sys
import time

import pytest
import torch
import torch.nn.functional as F

from artist_style_transfer_b200 import conv_geometry as cg
from test_geometry import _stack_filter, pack
from test_param_grad_kernels import _build, _window

CONV_RELU, CONV_REFLECT, CONV_ROUND_TF32 = 1, 2, 8      # include/ast.h AST_CONV_*
F16_MAX = 65504.0


# ---------------------------------------------------------------------------------------------------------------------
# fp64 references (include/ast.h), computed on the tensors' own device.

def _grid_limits(h, w, oy0, ox0, soy, sox, mi, mj):
    """Grid rows / columns whose output pixel lies inside an h x w output (outputs outside are skipped)."""
    ilim = min(mi, (h - oy0 + soy - 1) // soy) if oy0 < h else 0
    jlim = min(mj, (w - ox0 + sox - 1) // sox) if ox0 < w else 0
    return max(ilim, 0), max(jlim, 0)


def _blocks(kind, launches, h, w):
    """The output blocks of one call as (oy0, ox0, soy, sox, ilim, jlim, si_y, si_x, [(dy, dx, weight key)], label).
    A conv_gather launch is one block whose taps read W[woff + t]; a conv_stacked call has nblk blocks whose taps are the
    virtual taps with a filter tile in that block (Ws[v][g*cb:(g+1)*cb])."""
    out = []
    if kind == "gather":
        for li, l in enumerate(launches):
            ilim, jlim = _grid_limits(h, w, l.oy0, l.ox0, l.so, l.so, l.mi, l.mj)
            taps = [(dy, dx, l.woff + t) for t, (dy, dx) in enumerate(l.taps)]
            out.append((l.oy0, l.ox0, l.so, l.so, ilim, jlim, l.si, l.si, taps, f"launch {li}"))
    else:
        stk = launches
        for g in range(stk.nblk):
            ilim, jlim = _grid_limits(h, w, stk.oy[g], stk.ox[g], stk.soy, stk.sox, stk.mi, stk.mj)
            taps = [(dy, dx, (v, g)) for v, (dy, dx) in enumerate(stk.vt) if stk.src[v][g] is not None]
            out.append((stk.oy[g], stk.ox[g], stk.soy, stk.sox, ilim, jlim, stk.sy, 1, taps, f"block {g}"))
    return out


def written_mask(kind, launches, h, w, device):
    """[h, w] bool: the output pixels a call's launches (or blocks) map into its output."""
    m = torch.zeros(h, w, dtype=torch.bool, device=device)
    for oy0, ox0, soy, sox, ilim, jlim, *_ in _blocks(kind, launches, h, w):
        if ilim and jlim:
            m[oy0 + soy * torch.arange(ilim, device=device)[:, None], ox0 + sox * torch.arange(jlim, device=device)] = True
    return m


def _weight(kind, w, key, n, cout, w_img_stride):
    """fp64 [cout][cin] weights of one tap for image n."""
    if kind == "gather":
        cpad, cin = w.shape[-2], w.shape[-1]           # packed rows per tap (ops.conv_gather strides launches by them)
        flat = w.reshape(-1)
        off = n * w_img_stride + key * cpad * cin
        return flat[off:off + cpad * cin].view(cpad, cin)[:cout].double()
    v, g = key
    return w[v, g * cout:(g + 1) * cout].double()


def epilogue(pre, bias=None, add=None, mask=None, relu=False):
    """tc_epilogue32 (csrc/tc_common.cuh) in fp64: bias -> add -> ReLU -> mask (mask > 0).  The TF32 rounding and the store
    are the output rounding of the error bound."""
    v = pre
    if bias is not None:
        v = v + bias.double()
    if add is not None:
        v = v + add.double()
    if relu:
        v = v.clamp_min(0)
    if mask is not None:
        v = torch.where(mask > 0, v, torch.zeros_like(v))
    return v


def _contract(kind, x, w, launches, out_shape, in_shift, w_img_stride, lo, hi, with_rows=False):
    """pre / A ([hi-lo, H, W, cout] fp64, NaN / 0 outside the written set) and, with_rows, the contribution of every tap to
    the last grid row of the last image that has a non-zero one, in the last block that has such a row (for the tap
    mutant; the last rows of some phases read only the zero border of a data gradient)."""
    _, h, w_, cout = out_shape
    nc = hi - lo
    dev = x.device
    x64 = x[lo:hi].double()
    if in_shift is not None:
        x64 = x64 + in_shift.double()          # _window zeroes out-of-range pixels afterwards: the shift reaches in-range ones
    pre = torch.full((nc, h, w_, cout), float("nan"), dtype=torch.float64, device=dev)
    A = torch.zeros((nc, h, w_, cout), dtype=torch.float64, device=dev)
    rows = None
    blocks = [b for b in _blocks(kind, launches, h, w_) if b[4] and b[5]]
    for bi, (oy0, ox0, soy, sox, ilim, jlim, sy, sx, taps, label) in enumerate(blocks):
        acc = torch.zeros((nc, ilim, jlim, cout), dtype=torch.float64, device=dev)
        acca = torch.zeros_like(acc)
        tapw = []
        for dy, dx, key in taps:
            xt = _window(x64, dy, dx, sy, sx, ilim, jlim)                         # [nc, ilim, jlim, cin]
            if w_img_stride:
                wt = torch.stack([_weight(kind, w, key, lo + i, cout, w_img_stride) for i in range(nc)])
                acc += torch.matmul(xt.flatten(1, 2), wt.transpose(1, 2)).view_as(acc)
                acca += torch.matmul(xt.abs().flatten(1, 2), wt.abs().transpose(1, 2)).view_as(acc)
                wl = wt[-1]
            else:
                wt = _weight(kind, w, key, 0, cout, 0)
                acc += xt @ wt.t()
                acca += xt.abs() @ wt.abs().t()
                wl = wt
            tapw.append((dy, dx, key, wl))
            del xt
        ys = oy0 + soy * torch.arange(ilim, device=dev)
        xs = ox0 + sox * torch.arange(jlim, device=dev)
        pre[:, ys[:, None], xs[None, :]] = acc
        A[:, ys[:, None], xs[None, :]] = acca
        for i in reversed(range(ilim)) if with_rows else ():
            contrib = [((dy, dx, key), _window(x64[-1:], sy * i + dy, dx, sy, sx, 1, jlim)[0, 0] @ wl.t())
                       for dy, dx, key, wl in tapw]                                 # [jlim, cout] per tap
            if any(float(c.abs().max()) > 0 for _, c in contrib):
                rows = dict(y=int(ys[i]), xs=xs, contrib=contrib, label=label)
                break
    return pre, A, rows


def conv_reference(kind, x, w, launches, out_shape, bias=None, in_shift=None, add=None, mask=None, flags=0,
                   w_img_stride=0, images=None, mutants=False):
    """fp64 reference of one `ast_conv_gather` (kind "gather": w = packed [taps][cpad][cin], launches = [Launch]) or
    `ast_conv_stacked` (kind "stacked": w = [nvt][128][cin], launches = conv_geometry.Stacked) call, for images
    [lo, hi) = `images` (default: all).  add / mask: the call's full images.  Returns a dict of [hi-lo, H, W, cout] fp64:
      ref   the pre-store values (NaN outside the written set);
      A     the same contraction of |x| and |W| (+ |bias| + |add|), masked like ref: the scale of the error bound;
      pre   the sums before bias (InstanceNorm statistics);
    and, with `mutants` (the chunk must hold the last image), `mutants` = {name: (ref-shaped tensor, description)}:
      tap      ref without one tap's contribution on the last grid row of the last image that has a non-zero one
               (the tap with the smallest non-zero contribution there), i.e. a kernel that lost a halo column / edge tile there;
      wrong_image (per-image weights) the last image computed with the weights of the image whose weights differ most
               from its own (the Gram backward weights of iid noise images agree to ~1e-4, less than a bf16 rounding:
               such a mutant is printed but cannot be required to fail);
      no_add   (with add) ref without the add;  no_mask (with mask) ref without the mask."""
    assert not flags & CONV_REFLECT, "no production call mirrors out-of-range coordinates in a convolution"
    n = out_shape[0]
    lo, hi = images or (0, n)
    relu = bool(flags & CONV_RELU)
    pre, A, rows = _contract(kind, x, w, launches, out_shape, in_shift, w_img_stride, lo, hi, with_rows=mutants)
    a_ = None if add is None else add[lo:hi]
    m_ = None if mask is None else mask[lo:hi]
    ref = epilogue(pre, bias, a_, m_, relu)
    scale = A + (0 if bias is None else bias.double().abs()) + (0 if a_ is None else a_.double().abs())
    if m_ is not None:
        scale = torch.where(m_ > 0, scale, torch.zeros_like(scale))
    res = dict(ref=ref, A=scale, pre=pre, A_pre=A)
    if not mutants:
        return res
    assert hi == n
    mut = {}
    if rows is not None:
        nz = [(float(c.norm()), k, c) for k, c in rows["contrib"] if float(c.norm()) > 0]
        if nz:
            _, key, c = min(nz, key=lambda t: t[0])
            p = pre.clone()
            p[-1, rows["y"], rows["xs"]] -= c
            mut["tap"] = (epilogue(p, bias, a_, m_, relu), f"tap {key} of {rows['label']} on output row {rows['y']}")
    if w_img_stride and n > 1:
        sets = w.reshape(-1)[:n * w_img_stride].view(n, w_img_stride).double()
        k = int((sets[:-1] - sets[-1]).norm(dim=1).argmax())
        wk = sets[k].view(-1, w.shape[-2], w.shape[-1])                        # image k's set as shared weights
        pk, _, _ = _contract(kind, x[n - 1:n], wk, launches, (1,) + tuple(out_shape[1:]), in_shift, 0, 0, 1)
        p = pre.clone()
        p[-1] = pk[0]
        dw = float((sets[k] - sets[-1]).norm() / sets[-1].norm())
        mut["wrong_image"] = (epilogue(p, bias, a_, m_, relu), f"last image with image {k}'s weights", dw)
    if a_ is not None:
        mut["no_add"] = (epilogue(pre, bias, None, m_, relu), "without add")
    if m_ is not None:
        mut["no_mask"] = (epilogue(pre, bias, a_, None, relu), "without mask")
    res["mutants"] = mut
    return res


def pool_reference(t):
    """nn.MaxPool2d(2, 2) of an NHWC tensor and the pool_codes byte of include/ast.h: bits 0-1 = arg max k = 2*dy + dx
    (the first maximum wins), bits 2-5 = (x_k > 0)."""
    h, w = t.shape[1] // 2 * 2, t.shape[2] // 2 * 2
    win = [t[:, dy:h:2, dx:w:2] for dy in (0, 1) for dx in (0, 1)]
    m = win[0]
    arg = torch.zeros(m.shape, dtype=torch.uint8, device=t.device)
    for k in (1, 2, 3):
        gt = win[k] > m
        m = torch.where(gt, win[k], m)
        arg = torch.where(gt, torch.full_like(arg, k), arg)
    code = arg
    for k in range(4):
        code = code | ((win[k] > 0).to(torch.uint8) << (2 + k))
    return m, code


def _reflect(i, n):
    i = i.abs()
    return torch.where(i >= n, 2 * (n - 1) - i, i)


def round_tf32(t):
    """cvt.rna.tf32.f32 of an fp32 tensor: keep 10 mantissa bits, round half away from zero."""
    b = t.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def row_im2col_reference(src, out_shape, out_dtype, kw, sign, px, py, reflect, shift=None, rnd=False):
    """ast_row_im2col: out[n, y, x, d*C + c] = src[n, Y(y - py), X(x + sign*d - px), c] (+ shift[c]) for d < kw, channels
    kw*C .. out.c - 1 zero.  Out-of-range coordinates are mirrored (reflect) or read 0 - the shift is applied before the
    zero padding, so padded pixels are 0, not shift.  Computed in fp32 like the kernel, then stored in out_dtype."""
    n, h, w, c = src.shape
    _, ho, wo, oc = out_shape
    dev = src.device
    s = src.float()
    if shift is not None:
        s = s + shift.float()
    out = torch.zeros((n, ho, wo, oc), dtype=torch.float32, device=dev)
    ys = torch.arange(ho, device=dev) - py
    for d in range(kw):
        xs = torch.arange(wo, device=dev) + sign * d - px
        if reflect:
            out[..., d * c:(d + 1) * c] = s[:, _reflect(ys, h)][:, :, _reflect(xs, w)]
        else:
            out[..., d * c:(d + 1) * c] = _window(s, int(ys[0]), int(xs[0]), 1, 1, ho, wo)
    if rnd:
        out = round_tf32(out)
    return out.to(out_dtype)


def fold_rows_reference(part, out_shape, kw, bias=None, relu=False):
    """ast_fold_rows in fp64: out[n, y, x, c] = bias[c] + sum_{d < kw} part[n, y, x + d, d*C + c] (ReLU).  Also returns
    sum |terms| + |bias|, the scale of the fp32 sum's rounding."""
    _, h, w, c = out_shape
    p = part.double()
    ref = torch.zeros(out_shape, dtype=torch.float64, device=part.device)
    scale = torch.zeros_like(ref)
    for d in range(kw):
        t = p[:, :h, d:d + w, d * c:(d + 1) * c]
        ref += t
        scale += t.abs()
    if bias is not None:
        ref += bias.double()
        scale += bias.double().abs()
    if relu:
        ref = ref.clamp_min(0)
    return ref, scale


# ---------------------------------------------------------------------------------------------------------------------
# CPU checks of the references.

def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("k,s,pad,h,w", [(3, 1, 1, 9, 11), (3, 2, 0, 13, 10), (9, 1, 0, 14, 12), (1, 1, 0, 5, 6)])
def test_reference_conv_fwd(k, s, pad, h, w):
    """conv_fwd launches (zero padding read as out-of-range, stride 2 at odd sizes) and the A scale on |x|, |W|."""
    torch.manual_seed(k * 10 + s + h)
    x = torch.randn(2, 5, h, w, dtype=torch.float64)
    wt = torch.randn(7, 5, k, k, dtype=torch.float64)
    want = F.conv2d(x, wt, stride=s, padding=pad)
    ls = cg.conv_fwd(k, s, pad, h, w)
    r = conv_reference("gather", _nhwc(x), pack(wt, ls, 0, 1), ls, _nhwc(want).shape)
    assert _rel(r["ref"], _nhwc(want)) < 1e-13
    assert _rel(r["A"], _nhwc(F.conv2d(x.abs(), wt.abs(), stride=s, padding=pad))) < 1e-13


@pytest.mark.parametrize("s,h,w", [(2, 11, 9), (2, 12, 14), (1, 8, 7)])
def test_reference_conv_dgrad(s, h, w):
    """conv_dgrad launches (stride-2 output phases) against torch.nn.grad.conv2d_input."""
    torch.manual_seed(20 + s + h)
    wt = torch.randn(6, 4, 3, 3, dtype=torch.float64)
    ho, wo = cg.conv_out_size(h, 3, s, 0), cg.conv_out_size(w, 3, s, 0)
    gy = torch.randn(2, 6, ho, wo, dtype=torch.float64)
    want = torch.nn.grad.conv2d_input((2, 4, h, w), wt, gy, stride=s)
    ls = cg.conv_dgrad(3, s, 0, h, w)
    r = conv_reference("gather", _nhwc(gy), pack(wt, ls, 1, 0), ls, (2, h, w, 4))
    assert _rel(r["ref"], _nhwc(want)) < 1e-13
    wa = torch.nn.grad.conv2d_input((2, 4, h, w), wt.abs(), gy.abs(), stride=s)
    assert _rel(r["A"], _nhwc(wa)) < 1e-13


@pytest.mark.parametrize("k,s,op,h,w", [(3, 2, 1, 6, 7), (1, 1, 0, 5, 4)])
def test_reference_conv_transpose_fwd_and_dgrad(k, s, op, h, w):
    """convT_fwd (sub-pixel phases) and convT_dgrad against conv_transpose2d and its input gradient."""
    torch.manual_seed(30 + k)
    x = torch.randn(2, 4, h, w, dtype=torch.float64, requires_grad=True)
    wt = torch.randn(4, 6, k, k, dtype=torch.float64)
    y = F.conv_transpose2d(x, wt, stride=s, padding=k // 2, output_padding=op)
    ls = cg.convT_fwd(k, s, k // 2, op, h, w)
    r = conv_reference("gather", _nhwc(x.detach()), pack(wt, ls, 1, 0), ls, _nhwc(y).shape)
    assert _rel(r["ref"], _nhwc(y.detach())) < 1e-13
    wa = F.conv_transpose2d(x.detach().abs(), wt.abs(), stride=s, padding=k // 2, output_padding=op)
    assert _rel(r["A"], _nhwc(wa)) < 1e-13
    gy = torch.randn_like(y)
    (gx,) = torch.autograd.grad(y, x, gy)
    ld = cg.convT_dgrad(k, s, k // 2, y.shape[2], y.shape[3])
    rd = conv_reference("gather", _nhwc(gy), pack(wt, ld, 0, 1), ld, (2, h, w, 4))
    assert _rel(rd["ref"], _nhwc(gx)) < 1e-13


@pytest.mark.parametrize("sign", [1, -1])
def test_reference_vertical_taps(sign):
    """A 9-tap vertical launch (the row-folded ends; sign -1: the thin-output data gradient reading rows y - d)."""
    torch.manual_seed(40)
    n, h, w, cin, cout = 2, 13, 6, 5, 3
    x = torch.randn(n, h, w, cin, dtype=torch.float64)
    wt = torch.randn(cout, cin, 9, 1, dtype=torch.float64)
    taps = [(sign * d, 0) for d in range(9)]
    ho = h - 8 if sign == 1 else h + 8
    ls = [cg.Launch(ho, w, 1, 1, 0, 0, taps, [(d, 0) for d in range(9)], 0)]
    r = conv_reference("gather", x, pack(wt, ls, 0, 1), ls, (n, ho, w, cout))
    xin = x.permute(0, 3, 1, 2)
    want = F.conv2d(xin, wt) if sign == 1 else F.conv2d(F.pad(xin, (0, 0, 8, 8)), wt.flip(2))
    assert _rel(r["ref"], _nhwc(want)) < 1e-13


def test_reference_per_image_weights():
    """The Gram backward: one tap, per-image C x C weights (w_img_stride), against torch.bmm."""
    torch.manual_seed(41)
    n, h, w, c = 3, 5, 7, 8
    x = torch.randn(n, h, w, c, dtype=torch.float64)
    d = torch.randn(n, c, c, dtype=torch.float64)
    ls = cg.conv_fwd(1, 1, 0, h, w)
    r = conv_reference("gather", x, d.view(n, 1, c, c), ls, (n, h, w, c), w_img_stride=c * c, mutants=True)
    want = torch.bmm(x.view(n, h * w, c), d.transpose(1, 2)).view(n, h, w, c)
    assert _rel(r["ref"], want) < 1e-13
    wa = torch.bmm(x.abs().view(n, h * w, c), d.abs().transpose(1, 2)).view(n, h, w, c)
    assert _rel(r["A"], wa) < 1e-13
    k = int((d[:-1] - d[-1]).flatten(1).norm(dim=1).argmax())
    mk = torch.bmm(x[-1:].view(1, h * w, c), d[k:k + 1].transpose(1, 2)).view(1, h, w, c)
    assert _rel(r["mutants"]["wrong_image"][0][-1], mk[0]) < 1e-13
    assert abs(r["mutants"]["wrong_image"][2] - _rel(d[k], d[-1])) < 1e-12
    assert torch.equal(r["mutants"]["wrong_image"][0][:-1], r["ref"][:-1])


def test_reference_in_shift_on_a_zero_padded_input():
    """VGG conv1_1 in strict mode: the mean shift is added to in-range pixels only, then the zero padding."""
    torch.manual_seed(42)
    x = torch.rand(2, 3, 9, 10, dtype=torch.float64) * 255
    shift = torch.tensor([-103.939, -116.779, -123.68], dtype=torch.float64)
    wt = torch.randn(4, 3, 3, 3, dtype=torch.float64)
    ls = cg.conv_fwd(3, 1, 1, 9, 10)
    r = conv_reference("gather", _nhwc(x), pack(wt, ls, 0, 1), ls, (2, 9, 10, 4), in_shift=shift)
    want = F.conv2d(x + shift.view(1, 3, 1, 1), wt, padding=1)
    assert _rel(r["ref"], _nhwc(want)) < 1e-13
    wa = F.conv2d((x + shift.view(1, 3, 1, 1)).abs(), wt.abs(), padding=1)
    assert _rel(r["A"], _nhwc(wa)) < 1e-13


def test_reference_epilogue_bias_add_relu_mask():
    """bias -> add -> ReLU -> (mask > 0), and A = (|x|*|W| + |bias| + |add|) where the mask passes."""
    torch.manual_seed(43)
    x = torch.randn(2, 4, 8, 9, dtype=torch.float64)
    wt = torch.randn(5, 4, 3, 3, dtype=torch.float64)
    b = torch.randn(5, dtype=torch.float64)
    add = torch.randn(2, 8, 9, 5, dtype=torch.float64)
    mask = torch.randn(2, 8, 9, 5, dtype=torch.float64)
    ls = cg.conv_fwd(3, 1, 1, 8, 9)
    r = conv_reference("gather", _nhwc(x), pack(wt, ls, 0, 1), ls, (2, 8, 9, 5), bias=b, add=add, mask=mask,
                       flags=CONV_RELU, mutants=True)
    conv = _nhwc(F.conv2d(x, wt, padding=1))
    want = torch.where(mask > 0, (conv + b + add).clamp_min(0), torch.zeros_like(conv))
    assert _rel(r["ref"], want) < 1e-13
    wa = torch.where(mask > 0, _nhwc(F.conv2d(x.abs(), wt.abs(), padding=1)) + b.abs() + add.abs(), torch.zeros_like(conv))
    assert _rel(r["A"], wa) < 1e-13
    assert _rel(r["pre"], conv) < 1e-13
    assert _rel(r["mutants"]["no_add"][0], torch.where(mask > 0, (conv + b).clamp_min(0), torch.zeros_like(conv))) < 1e-13
    assert _rel(r["mutants"]["no_mask"][0], (conv + b + add).clamp_min(0)) < 1e-13


def test_reference_tap_mutant_is_one_tap_less_on_one_row():
    """The tap mutant equals the reference computed with that tap's weights zeroed, on that grid row of the last image
    (and the reference everywhere else)."""
    torch.manual_seed(44)
    n, h, w = 2, 10, 12
    x = torch.randn(n, 4, h, w, dtype=torch.float64)
    wt = torch.randn(4, 6, 3, 3, dtype=torch.float64)
    ls = cg.convT_fwd(3, 2, 1, 1, h, w)
    wp = pack(wt, ls, 1, 0)
    shape = (n, 2 * h, 2 * w, 6)
    r = conv_reference("gather", _nhwc(x), wp, ls, shape, mutants=True)
    mut, what = r["mutants"]["tap"]
    diff = (mut != r["ref"]).any(-1)
    assert diff[:-1].sum() == 0
    rows = diff[-1].nonzero()[:, 0].unique()
    assert rows.numel() == 1, what
    y = int(rows[0])
    l = ls[-1]
    assert (y - l.oy0) % l.so == 0 and y == l.oy0 + l.so * (l.mi - 1)
    # the tap: the one whose removal reproduces the row
    hits = 0
    for t in range(len(l.taps)):
        wz = wp.clone()
        wz[l.woff + t] = 0
        rz = conv_reference("gather", _nhwc(x), wz, ls, shape)["ref"]
        xs = l.ox0 + l.so * torch.arange(l.mj)
        hits += int(torch.allclose(mut[-1, y, xs], rz[-1, y, xs], rtol=0, atol=1e-12))
    assert hits >= 1, what
    assert _rel(mut, r["ref"]) > 1e-4


@pytest.mark.parametrize("case", ["convT32", "dgrad32", "convT64", "rows9", "rows3_64", "rows9_neg", "rows3x3"])
def test_stacked_reference_equals_the_plain_launches(case):
    """conv_reference of a conv_stacked call equals conv_reference of the plain gather launches it replaces (the cases of
    test_geometry.test_stacked_launches_equal_the_plain_gather)."""
    torch.manual_seed(1)
    cb = 64 if "64" in case else 32
    if case in ("convT32", "convT64"):
        hin, win, ls, ho, wo = 7, 9, cg.convT_fwd(3, 2, 1, 1, 7, 9), 14, 18
    elif case == "dgrad32":
        hin, win, ho, wo = 6, 7, 14, 16
        ls = cg.conv_dgrad(3, 2, 0, ho, wo)
    elif case == "rows9":
        hin, win, ho, wo = 19, 10, 11, 10
        ls = [cg.Launch(ho, wo, 1, 1, 0, 0, [(d, 0) for d in range(9)], [(d, 0) for d in range(9)], 0)]
    elif case == "rows9_neg":
        hin, win, ho, wo = 10, 9, 18, 9
        ls = [cg.Launch(ho, wo, 1, 1, 0, 0, [(-d, 0) for d in range(9)], [(d, 0) for d in range(9)], 0)]
    elif case == "rows3_64":
        hin, win, ho, wo = 9, 8, 9, 8
        ls = [cg.Launch(ho, wo, 1, 1, 0, 0, [(-1, 0), (0, 0), (1, 0)], [(0, 0), (1, 0), (2, 0)], 0)]
    else:
        hin, win, ho, wo = 10, 11, 10, 11
        ls = cg.conv_fwd(3, 1, 1, hin, win)
    nt = sum(len(l.taps) for l in ls)
    x = torch.randn(2, hin, win, 6, dtype=torch.float64)
    wt = torch.randn(nt, cb, 6, dtype=torch.float64)
    b = torch.randn(cb, dtype=torch.float64)
    shape = (2, ho, wo, cb)
    want = conv_reference("gather", x, wt, ls, shape, bias=b, flags=CONV_RELU)
    nb = 128 // cb
    groups = [cg.stack_phases(ls[i:i + nb]) for i in range(0, len(ls), nb)] if len(ls) > 1 else [cg.stack_rows(ls[0], nb)]
    ref = torch.full(shape, float("nan"), dtype=torch.float64)
    a = torch.full(shape, float("nan"), dtype=torch.float64)
    for stk in groups:
        got = conv_reference("stacked", x, _stack_filter(wt, ls, stk, cb), stk, shape, bias=b, flags=CONV_RELU)
        wm = written_mask("stacked", stk, ho, wo, "cpu")
        assert not torch.isnan(got["ref"][:, wm]).any() and torch.isnan(got["ref"][:, ~wm]).all()
        ref[:, wm], a[:, wm] = got["ref"][:, wm], got["A"][:, wm]
    assert not torch.isnan(ref).any(), "the stacked calls do not cover the output"
    torch.testing.assert_close(ref, want["ref"], rtol=1e-13, atol=1e-13)
    torch.testing.assert_close(a, want["A"], rtol=1e-13, atol=1e-13)


def test_pool_reference_matches_max_pool2d():
    """Max and codes against F.max_pool2d(return_indices=True), with ties (first maximum wins) and all-negative windows."""
    torch.manual_seed(45)
    x = torch.randn(2, 6, 8, 10, dtype=torch.float32)
    x[0, :, :4] = x[0, :, :4].round()                       # many ties
    x[1, :, 4:] = -x[1, :, 4:].abs() - 0.5                  # all-negative windows
    x[1, 0, :2, :2] = 2.0                                   # a four-way tie: arg max 0
    m, idx = F.max_pool2d(x, 2, 2, return_indices=True)
    got_m, code = pool_reference(_nhwc(x))
    assert torch.equal(got_m, _nhwc(m))
    w = x.shape[3]
    k = ((idx // w) % 2) * 2 + (idx % w) % 2
    assert torch.equal((code & 3).long(), _nhwc(k))
    for kk, (dy, dx) in enumerate([(0, 0), (0, 1), (1, 0), (1, 1)]):
        assert torch.equal(((code >> (2 + kk)) & 1).bool(), _nhwc(x[:, :, dy::2, dx::2] > 0))
    assert int(code[1, 0, 0, 0]) & 3 == 0
    assert bool((code[1, 2:] >> 2 == 0).all())             # all-negative: no sign bit set


@pytest.mark.parametrize("reflect,sign,shift", [(True, 1, False), (False, 1, True), (False, -1, False)])
def test_row_im2col_reference(reflect, sign, shift):
    """The thin-input first layer (reflect), VGG conv1_1 (zero padding after the mean shift) and the thin-output filter
    gradient operand (sign -1): the row-folded image under a vertical convolution equals the plain convolution, and the
    channels beyond kw*C are zero."""
    torch.manual_seed(46)
    n, c, h, w, k = 2, 3, 9, 11, 3
    x = torch.rand(n, c, h, w) * 255
    sh = torch.tensor([-103.939, -116.779, -123.68]) if shift else None
    p = k // 2
    if sign == 1:
        out_shape = (n, h + 2 * p if reflect else h, w, 16)
        py = p if reflect else 0
        got = row_im2col_reference(_nhwc(x), out_shape, torch.float32, k, 1, p, py, reflect, shift=sh)
        xs = x + sh.view(1, 3, 1, 1) if shift else x
        full = F.pad(xs, (p, p, p, p), mode="reflect") if reflect else F.pad(xs, (p, p, 0, 0))
        for d in range(k):
            assert torch.equal(got[..., d * c:(d + 1) * c], _nhwc(full[..., d:d + w]))
    else:
        out_shape = (n, h, w + 2 * p, 16)
        got = row_im2col_reference(_nhwc(x), out_shape, torch.float32, k, -1, 0, 0, False)
        full = F.pad(x, (k - 1, k - 1, 0, 0))
        for d in range(k):
            assert torch.equal(got[..., d * c:(d + 1) * c], _nhwc(full[..., k - 1 - d:k - 1 - d + w + 2 * p]))
    assert float(got[..., k * c:].abs().sum()) == 0.0
    r = row_im2col_reference(_nhwc(x) * 1.0001, out_shape, torch.float32, k, sign, 1, 0, False, rnd=True)
    assert torch.equal(r, round_tf32(r)) and (r.view(torch.int32) & 0x1FFF).sum() == 0


def test_fold_rows_reference():
    """Horizontal taps computed as kw*C output channels of a vertical convolution, folded: equals the k x k convolution."""
    torch.manual_seed(47)
    n, cin, h, w, k, c = 2, 4, 7, 9, 3, 3
    x = torch.randn(n, cin, h + k - 1, w + k - 1, dtype=torch.float64)
    wt = torch.randn(c, cin, k, k, dtype=torch.float64)
    b = torch.randn(c, dtype=torch.float64)
    # part[n, y, x', d*C + co] = sum_{dy, ci} x[y + dy, x', ci] W[co, ci, dy, d]
    part = torch.zeros(n, h, w + k - 1, 32, dtype=torch.float64)
    for d in range(k):
        part[..., d * c:(d + 1) * c] = _nhwc(F.conv2d(x, wt[..., d:d + 1]))
    ref, scale = fold_rows_reference(part, (n, h, w, c), k, bias=b, relu=True)
    want = (F.conv2d(x, wt) + b.view(1, c, 1, 1)).clamp_min(0)
    assert _rel(ref, _nhwc(want)) < 1e-13
    assert bool((scale >= ref.abs()).all())


# ---------------------------------------------------------------------------------------------------------------------
# The real calls of a real step.

# Element-wise bound of one call:  |got - ref| <= tau * A + r * |ref| + floor.
#   tau, the accumulation error relative to A = sum |x|*|W| (+ |bias| + |add|):
#     strict (conv_simt, FFMA with fp32 operands, K = taps * cin <= 4608): each of the K fp32 roundings of the running sum
#       is <= 2^-24 of a partial sum <= A; a worst case of K * 2^-24 is never approached (errors of a sum of rounding
#       errors grow like sqrt(K)): tau = 2^-16.
#     fast, bf16 / fp16 operands (kind::f16, fp32 TMEM accumulation that truncates at every accumulate step, about
#       K/8 * 2^-25 of the sum, DESIGN section 3): tau = 2^-13.
#     fast, fp32 operands (kind::tf32: the Gram backward, whose x side is TF32-rounded but whose weights D are not): the
#       MMA truncates D to 10 mantissa bits, 2^-10 of each product: tau = 2^-13 + 2^-10.
#   r, the rounding of the store: bf16 2^-8 (8 significant bits: round to nearest is within half an ulp, 2^-8 of the
#     value - the 2^-9 of the first draft of these bounds was an ulp of the wrong size and fails on ties), fp16 and TF32
#     (cvt.rna) 2^-11, fp32 0.  fp16 stores saturate: fp16 outputs are compared with the reference clamped to +-65504.
#   floor: fp16 subnormals are spaced 2^-24 apart (half of it is the rounding); bf16 and fp32 have fp32's exponent range.
# Whole output: ||got - ref|| <= r * ||ref|| + eps * ||A|| with eps = tau / 16: rounding errors do not share a sign, so the
#   norm of the error stays far below tau * ||A|| (which the element bound alone would allow).
CONV_TAU = {"fp32": 2.0 ** -16, "fast": 2.0 ** -13}
TF32_OPERAND = 2.0 ** -10
OUT_ROUND = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
OUT_FLOOR = {torch.float32: 0.0, torch.bfloat16: 0.0, torch.float16: 2.0 ** -25}
FRO_EPS = 1.0 / 16
# The fused InstanceNorm statistics: each stored value v differs from the fp64 pre-bias sum by at most tau * A_pre; the
# kernels add v and (v - mu)^2 of <= 32 pixels in fp32 before the fp64 accumulation (<= 32 roundings of 2^-24 of a partial
# sum <= sum |v| resp. sum v^2): |d sum x| <= tau * sum A + 2^-19 * sum |x|, |d sum x^2| <= 2 tau * sum A*|x| + 2^-19 * sum x^2
# (+ tau^2 * sum A^2, negligible, covered by a factor 2).  tau here is calibrated, not the element model: with tau = 2^-13
# the largest |d stats| / bound measured on a B200 over the five workloads below was 4.5e-4 (the statistics come from the
# fp32 accumulators, before any output rounding), a bound so loose that sum x^2 without one grid row of a 1024^2 plane
# passed it.  STATS_TAU = 2^-19 is 64x tighter and still leaves 35x margin over the measurement.
STATS_TAU = 2.0 ** -19
STATS_PARTIAL = 2.0 ** -19
CONV_FAMILIES = ("conv_tc", "conv_px", "conv_ws", "conv_hx", "conv_st", "conv_simt")
# DESIGN section 5: conv launches of one step at B = 32, 256^2, fast mode
STEP_FAMILIES_B32 = {"conv_hx": 37, "conv_st": 12, "conv_ws": 8, "conv_px": 5, "conv_tc": 3}
CHUNK_BYTES = 1 << 30           # fp64 working set of one reference chunk


def _storage_view(t):
    """The whole storage under t as a flat tensor of t's dtype."""
    esz = t.element_size()
    return torch.empty(0, dtype=t.dtype, device=t.device).set_(t.untyped_storage(), 0, (t.untyped_storage().nbytes() // esz,),
                                                                (1,))


def _bits(t):
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def _changed_outside(before, after, inside):
    return int(((_bits(before) != _bits(after)) & ~inside).sum())


def _inside(t, sel):
    """bool over t's storage: True at the elements of t selected by sel(view) (a function applied to a bool view)."""
    st = _storage_view(t)
    ins = torch.zeros(st.shape, dtype=torch.bool, device=t.device)
    sel(ins.as_strided(t.shape, t.stride(), t.storage_offset()))
    return ins


def _site():
    """file:line of the library code that made the call (cnn.py / train_cnn.py), for the printout."""
    f = sys._getframe(2)
    while f is not None:
        fn = os.path.basename(f.f_code.co_filename)
        if fn in ("cnn.py", "train_cnn.py"):
            return f"{fn}:{f.f_lineno}"
        f = f.f_back
    return "?"


class _ConvProbe:
    """Wraps ops.conv_gather / conv_stacked / row_im2col / fold_rows.  Each call: NaN in the positions it must write,
    snapshots of the rest of its output's storage and of its side outputs, clones of its inputs, family counters; then the
    real call with unchanged arguments, a synchronise, the fp64 reference and a record.  Asserts come after the step."""

    NAMES = ("conv_gather", "conv_stacked", "row_im2col", "fold_rows")

    def __init__(self, lib, ops, mode):
        self.lib, self.mode = lib, mode
        self.real = {name: getattr(ops, name) for name in self.NAMES}
        self.conv, self.helpers = [], []

    def _bind(self, name, args, kwargs):
        a = inspect.signature(self.real[name]).bind(*args, **kwargs)
        a.apply_defaults()
        return a.arguments

    def _run(self, name, args, kwargs):
        fam0 = self.lib.family_stats()
        res = self.real[name](*args, **kwargs)
        torch.cuda.synchronize()
        return res, self.lib.family_delta(fam0)

    def conv_gather(self, *args, **kwargs):
        a = self._bind("conv_gather", args, kwargs)
        flags = (CONV_RELU if a["relu"] else 0) | (CONV_REFLECT if a["reflect"] else 0)
        return self._conv("conv_gather", "gather", args, kwargs, a["x"], a["wpacked"], a["launches"], a["out"], a["bias"],
                          a["in_shift"], a["add"], a["mask"], flags, a["w_img_stride"], a["round_tf32"], a["stats"],
                          a["pooled"], a["pool_codes"], a["pool_only"])

    def conv_stacked(self, *args, **kwargs):
        a = self._bind("conv_stacked", args, kwargs)
        return self._conv("conv_stacked", "stacked", args, kwargs, a["x"], a["wstacked"], a["stk"], a["out"], a["bias"],
                          None, a["add"], a["mask"], CONV_RELU if a["relu"] else 0, 0, a["round_tf32"], a["stats"],
                          None, None, False)

    def _conv(self, name, kind, args, kwargs, x, w, launches, out, bias, in_shift, add, mask, flags, wis, rnd, stats,
              pooled, codes, pool_only):
        n, h, wd, cout = out.shape
        dev = out.device
        wm = written_mask(kind, launches, h, wd, dev)
        if not pool_only:
            out[:, wm] = float("nan")
        st_out = _storage_view(out)
        before_out = st_out.clone()
        side = {}
        if pooled is not None:
            pooled.fill_(float("nan"))
            side["pooled"] = pooled
        if codes is not None:
            codes.fill_(255)                        # bits 6-7 set: never a valid window code
            side["codes"] = codes
        if stats is not None:
            side["stats"] = stats
        side_before = {k: _storage_view(t).clone() for k, t in side.items()}
        stats_before = None if stats is None else stats.clone()
        inputs = {k: t for k, t in dict(x=x, w=w, bias=bias, in_shift=in_shift, add=add, mask=mask).items() if t is not None}
        clones = {k: t.clone() for k, t in inputs.items()}

        res, fam = self._run(name, args, kwargs)

        rec = dict(entry=name, site=_site(), kind=kind, x=(tuple(x.shape), str(x.dtype)[6:]), out=(tuple(out.shape),
                   str(out.dtype)[6:]), wdtype=str(w.dtype)[6:], n_launch=len(launches) if kind == "gather" else 1,
                   fams={f: fam[f][0] for f in CONV_FAMILIES if fam[f][0]}, pool_only=pool_only,
                   flags=dict(relu=bool(flags & CONV_RELU), bias=bias is not None, add=add is not None,
                              mask=mask is not None, tf32=bool(rnd), stats=stats is not None, pooled=pooled is not None,
                              per_image=bool(wis)))
        rec["inputs_changed"] = [k for k, t in inputs.items() if not torch.equal(_bits(t), _bits(clones[k]))]
        del clones
        # ---- coverage
        if pool_only:
            rec["changed_outside"] = _changed_outside(before_out, st_out, torch.zeros_like(st_out, dtype=torch.bool))
            rec["nan_left"] = 0
        else:
            ins = _inside(out, lambda v: v.__setitem__((slice(None), wm), True))
            rec["changed_outside"] = _changed_outside(before_out, st_out, ins)
            rec["nan_left"] = int(torch.isnan(out[:, wm]).sum())
            del ins
        del before_out
        for k, t in side.items():
            if k == "stats":
                ins = _inside(t, lambda v: v.fill_(True))
                rec["stats_changed_outside"] = _changed_outside(side_before[k], _storage_view(t), ins)
        del side_before
        # ---- values, chunk by chunk
        tau = CONV_TAU[self.mode] + (TF32_OPERAND if self.mode == "fast" and x.dtype == torch.float32 else 0.0)
        r = 2.0 ** -11 if rnd else OUT_ROUND[out.dtype]
        floor = OUT_FLOOR[out.dtype]
        rec.update(tau=tau, r=r)
        per_img = h * wd * max(x.shape[3], cout) * 8 * 4
        step = max(1, min(n, CHUNK_BYTES // per_img))
        err2 = ref2 = a2 = 0.0
        max_ratio = max_excess = 0.0
        bad = 0
        mut = {}
        s_ref = torch.zeros((n, cout, 2), dtype=torch.float64, device=dev)
        s_bound = torch.zeros_like(s_ref)
        s_mut = None
        pool_bad = pool_max = None
        for lo in range(0, n, step):
            hi = min(n, lo + step)
            R = conv_reference(kind, x, w, launches, out.shape, bias, in_shift, add, mask, flags, wis, (lo, hi),
                               mutants=hi == n)
            ref, A = R["ref"][:, wm], R["A"][:, wm]                      # [nc, P, cout]
            cmp = ref.clamp(-F16_MAX, F16_MAX) if out.dtype == torch.float16 else ref
            bound = tau * A + r * cmp.abs() + floor
            if not pool_only:
                got = out[lo:hi][:, wm].double()
                err = (got - cmp).abs()
                bad += int((err > bound).sum())
                max_ratio = max(max_ratio, float((err / A.clamp_min(1e-300)).max()))
                max_excess = max(max_excess, float((err / bound.clamp_min(1e-300)).max()))
                err2 += float(err.square().sum())
                ref2 += float(cmp.square().sum())
                a2 += float(A.square().sum())
                for k, (m, what, *dw) in R.get("mutants", {}).items():
                    mm = m[:, wm].clamp(-F16_MAX, F16_MAX) if out.dtype == torch.float16 else m[:, wm]
                    mut[k] = (float(((got - mm).abs() / bound.clamp_min(1e-300)).max()), what, *dw)
            if stats is not None:
                pre, Ap = R["pre"][:, wm], R["A_pre"][:, wm]
                s_ref[lo:hi, :, 0] = pre.sum(1)
                s_ref[lo:hi, :, 1] = pre.square().sum(1)
                s_bound[lo:hi, :, 0] = 2 * (STATS_TAU * Ap.sum(1) + STATS_PARTIAL * pre.abs().sum(1))
                s_bound[lo:hi, :, 1] = 2 * (2 * STATS_TAU * (Ap * pre.abs()).sum(1) + STATS_PARTIAL * pre.square().sum(1))
                if hi == n:                                             # sum x^2 without the last grid row of the last image
                    rows = R["pre"][-1, :, :, :]
                    last_y = int(wm.any(1).nonzero().max())
                    row = rows[last_y][wm[last_y]]
                    s_mut = (s_ref[n - 1, :, 1] - row.square().sum(0))
            if pooled is not None and pool_only:
                pm, _ = pool_reference(R["ref"].clamp(-F16_MAX, F16_MAX))
                pb, _ = pool_reference(_full_bound(R, wm, bound))
                pg = pooled[lo:hi].double()
                e = (pg - pm).abs() / (pb + 2.0 ** -11 * pm.abs() + 2.0 ** -25)
                pool_bad = (pool_bad or 0) + int((e > 1).sum()) + int(torch.isnan(pg).sum())
                pool_max = max(pool_max or 0.0, float(e.max()))
            del R
        rec.update(bad=bad, max_ratio=max_ratio, max_excess=max_excess, mutants=mut)
        if not pool_only:
            rec.update(fro=(err2 ** 0.5) / max(ref2 ** 0.5, 1e-300),
                       fro_tol=r + FRO_EPS * tau * (a2 ** 0.5) / max(ref2 ** 0.5, 1e-300))
        if stats is not None:
            d = stats.double() - stats_before.double()
            d = d.view(n, cout, 2)
            e = (d - s_ref).abs()
            rec["stats_bad"] = int((e > s_bound).sum())
            rec["stats_excess"] = float((e / s_bound.clamp_min(1e-300)).max())
            rec["stats_mutant"] = float(((d[n - 1, :, 1] - s_mut).abs() / s_bound[n - 1, :, 1]).max())
        if pooled is not None:
            if pool_only:
                rec["pool"] = dict(bad=pool_bad, excess=pool_max)
            else:
                pm, pc = pool_reference(out)
                rec["pool"] = dict(pooled_mismatch=int((_bits(pooled) != _bits(pm.clamp(-F16_MAX, F16_MAX).to(pooled.dtype))).sum()),
                                   codes_mismatch=-1 if codes is None else int((codes != pc).sum()))
        self.conv.append(rec)
        return res

    def row_im2col(self, *args, **kwargs):
        a = self._bind("row_im2col", args, kwargs)
        src, out = a["src"], a["out"]
        out.fill_(float("nan"))
        clones = {k: a[k].clone() for k in ("src", "shift") if a[k] is not None}
        res, fam = self._run("row_im2col", args, kwargs)
        want = row_im2col_reference(src, out.shape, out.dtype, a["kw"], a["sign"], a["px"], a["py"], a["reflect"],
                                    a["shift"], a["round_tf32"])
        self.helpers.append(dict(entry="row_im2col", site=_site(), shape=tuple(out.shape), dtype=str(out.dtype)[6:],
                                 mismatch=int((_bits(out) != _bits(want)).sum()),
                                 pad_nonzero=int((out[..., a["kw"] * src.shape[3]:] != 0).sum()),
                                 inputs_changed=[k for k, t in clones.items() if not torch.equal(_bits(a[k]), _bits(t))],
                                 launches=fam["pointwise"][0]))
        return res

    def fold_rows(self, *args, **kwargs):
        a = self._bind("fold_rows", args, kwargs)
        part, out = a["part"], a["out"]
        assert not a["flip_channels"], "stylize() is not on the training path"
        out.fill_(float("nan"))
        st = _storage_view(out)
        before = st.clone()
        clones = {k: a[k].clone() for k in ("part", "bias") if a[k] is not None}
        res, fam = self._run("fold_rows", args, kwargs)
        ref, scale = fold_rows_reference(part, out.shape, a["kw"], a["bias"], a["relu"])
        bound = (a["kw"] + 1) * 2.0 ** -24 * scale + OUT_ROUND[out.dtype] * ref.abs()
        err = (out.double() - ref).abs()
        ins = _inside(out, lambda v: v.fill_(True))
        self.helpers.append(dict(entry="fold_rows", site=_site(), shape=tuple(out.shape), dtype=str(out.dtype)[6:],
                                 mismatch=int((~(err <= bound)).sum()),
                                 max_excess=float((err / bound.clamp_min(1e-300)).max()),
                                 changed_outside=_changed_outside(before, st, ins),
                                 inputs_changed=[k for k, t in clones.items() if not torch.equal(_bits(a[k]), _bits(t))],
                                 launches=fam["pointwise"][0]))
        return res


def _full_bound(R, wm, bound):
    """The element bound as a full [nc, H, W, C] tensor (0 outside the written set), for pooling it."""
    full = torch.zeros_like(R["ref"])
    full[:, wm] = bound
    return full


WORKLOADS = [
    ("fast", 32, 256, 256),     # the benchmark workload
    ("fast", 1, 1024, 1024),    # BASELINE config 5
    ("fp32", 4, 256, 256),      # BASELINE config 1
    ("fp32", 1, 1024, 1024),    # config 5 in strict mode
    ("fast", 2, 132, 140),      # a multiple of 4, not of 16: partial tiles, odd phase grids, interleaved-row tails
]


@pytest.fixture(scope="module")
def ast():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import artist_style_transfer_b200 as m
    return m


def _fmt_mut(mut):
    return ", ".join(f"{k} {v[0]:.1f}x" + (f" (weights differ by {v[2]:.1e})" if len(v) > 2 else "")
                     for k, v in sorted(mut.items())) or "-"


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch,h,w", WORKLOADS, ids=[f"{m}-b{b}-{h}x{w}" for m, b, h, w in WORKLOADS])
def test_conv_launches_of_a_step(ast, monkeypatch, mode, batch, h, w):
    from artist_style_transfer_b200 import _lib, ops
    from oracle import weights
    t0 = time.time()
    net, vgg = _build(ast, mode)
    content = weights.content_batch(batch, h, 2, width=w).cuda()
    style = ast.style_grams_single(vgg, weights.style_image(h, 2).cuda(), batch)
    probe = _ConvProbe(_lib, ops, mode)
    for name in probe.NAMES:
        monkeypatch.setattr(ops, name, getattr(probe, name))
    fam0 = _lib.family_stats()
    ast.perceptual_step(net, vgg, content, style)        # eager: the probes synchronise, which graph capture forbids
    torch.cuda.synchronize()
    step = _lib.family_delta(fam0)
    monkeypatch.undo()

    tag = f"{mode} B={batch} {h}x{w}"
    fails = []
    for i, rec in enumerate(probe.conv):
        fam = "/".join(f"{f}x{c}" for f, c in rec["fams"].items()) or "none"
        fl = ",".join(k for k, v in rec["flags"].items() if v)
        where = f"#{i} {rec['entry']} {rec['site']} ({fam})"
        line = (f"[{tag}] {where}: x{rec['x'][0]} {rec['x'][1]} -> {rec['out'][0]} {rec['out'][1]} [{fl}] ")
        if rec["pool_only"]:
            line += f"pool-only: pooled err/bound {rec['pool']['excess']:.2e}"
        else:
            line += (f"|err|/|ref| {rec['fro']:.2e} (bound {rec['fro_tol']:.1e}), max err/A {rec['max_ratio']:.2e} "
                     f"(tau {rec['tau']:.1e}), max err/bound {rec['max_excess']:.2e}; mutants {_fmt_mut(rec['mutants'])}")
        if rec["flags"]["stats"]:
            line += f"; stats err/bound {rec['stats_excess']:.2e}, row-less sum x^2 {rec['stats_mutant']:.1f}x"
        print(line)
        # family and launch count
        n_fam = sum(rec["fams"].values())
        want_n = rec["n_launch"]
        if n_fam != want_n:
            fails.append(f"{where}: expected {want_n} conv launches, counters say {rec['fams']}")
        if mode == "fast" and "conv_simt" in rec["fams"]:
            fails.append(f"{where}: fast mode ran the SIMT convolution")
        if mode == "fp32" and set(rec["fams"]) - {"conv_simt"}:
            fails.append(f"{where}: strict mode ran {rec['fams']}")
        if rec["entry"] == "conv_stacked" and set(rec["fams"]) - {"conv_st", "conv_hx"}:
            fails.append(f"{where}: a stacked call ran {rec['fams']}")
        # values
        if not rec["pool_only"]:
            if rec["bad"]:
                fails.append(f"{where}: {rec['bad']} elements over tau*A + r*|ref| (max err/bound {rec['max_excess']:.2e})")
            if not rec["fro"] <= rec["fro_tol"]:
                fails.append(f"{where}: whole-output error {rec['fro']:.2e} > {rec['fro_tol']:.2e}")
            want_mut = {"tap"} | ({"wrong_image"} if rec["flags"]["per_image"] and batch > 1 else set()) \
                | ({"no_add"} if rec["flags"]["add"] else set()) | ({"no_mask"} if rec["flags"]["mask"] else set())
            if set(rec["mutants"]) != want_mut:
                fails.append(f"{where}: mutants {sorted(rec['mutants'])}, expected {sorted(want_mut)}")
            for k, (v, what, *dw) in rec["mutants"].items():
                # images whose weights differ by less than the output rounding cannot be told apart in the output: the
                # Gram backward of iid noise images, whose weights agree to ~1e-4 (printed, not failed)
                if dw and dw[0] < 2 * rec["r"]:
                    continue
                if not v > 1:
                    fails.append(f"{where}: the mutant '{what}' stays within the bound ({v:.2f}x)")
        # coverage and inputs
        if rec["nan_left"]:
            fails.append(f"{where}: {rec['nan_left']} output elements of the written set were not written")
        if rec["changed_outside"]:
            fails.append(f"{where}: {rec['changed_outside']} elements of the output's storage outside the written set changed")
        if rec["inputs_changed"]:
            fails.append(f"{where}: inputs changed: {rec['inputs_changed']}")
        if rec["flags"]["stats"]:
            if rec["stats_bad"]:
                fails.append(f"{where}: {rec['stats_bad']} statistics off by more than the bound "
                             f"(max {rec['stats_excess']:.2e}x)")
            if rec["stats_changed_outside"]:
                fails.append(f"{where}: {rec['stats_changed_outside']} statistics of other layers changed")
            if not rec["stats_mutant"] > 1:
                fails.append(f"{where}: sum x^2 without one grid row stays within the bound ({rec['stats_mutant']:.2f}x)")
        if rec["flags"]["pooled"]:
            p = rec["pool"]
            if rec["pool_only"] and (p["bad"] or not p["excess"] <= 1):
                fails.append(f"{where}: pooled output off: {p}")
            if not rec["pool_only"] and (p["pooled_mismatch"] or p["codes_mismatch"]):
                fails.append(f"{where}: pooled / codes differ from the pooling of the stored output: {p}")
    for rec in probe.helpers:
        print(f"[{tag}] {rec['entry']} {rec['site']}: {rec['shape']} {rec['dtype']}: "
              + ", ".join(f"{k} {v}" for k, v in rec.items() if k not in ("entry", "site", "shape", "dtype")))
        if rec["mismatch"] or rec.get("pad_nonzero") or rec.get("changed_outside") or rec["inputs_changed"] \
                or rec["launches"] != 1:
            fails.append(f"{rec['entry']} {rec['site']}: {rec}")
    # launch accounting over the whole step: no convolution escapes the probe
    seen = {}
    for rec in probe.conv:
        for f, c in rec["fams"].items():
            seen[f] = seen.get(f, 0) + c
    ran = {f: step[f][0] for f in CONV_FAMILIES if step[f][0]}
    print(f"[{tag}] conv launches per family: {ran} ({sum(ran.values())} launches, {len(probe.conv)} calls); "
          f"wall time {time.time() - t0:.1f} s")
    if seen != ran:
        fails.append(f"the step ran conv launches {ran}, the probes saw {seen}")
    if (mode, batch, h, w) == ("fast", 32, 256, 256) and ran != STEP_FAMILIES_B32:
        fails.append(f"conv launches per family {ran}, DESIGN section 5 states {STEP_FAMILIES_B32}")
    assert probe.conv and not fails, "\n".join(fails)
