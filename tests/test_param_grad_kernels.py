"""Every launch of a training step that writes the TransformerNet gradient arena, against fp64 of its own operands.

The fused optimizer reads one flat fp32 gradient arena (arena.py).  Three kinds of kernel write it: the filter-gradient
contractions (`ast_wgrad_gather`: `wgrad_tc` / `wgrad_thin` on the tensor cores in fast mode, `wgrad_simt` in strict mode),
`ast_channel_sum` (bias of the last, norm-free layer) and `ast_batch_reduce` (every dgamma / dbeta).  The step-level
parity tests have to be loose (bf16 drift accumulates through 17 InstanceNorms), loose enough to miss a layer whose
filter gradient is a few per cent wrong.  Here a real `perceptual_step` runs with those three entry points wrapped: each
call snapshots the arena, runs once, and is compared with an fp64 evaluation of exactly the operands it received, so the
bounds are those of ONE fp32-accumulated contraction.  For every call the test also shows that the bound would catch the
loss of one grid row of one image (a dropped or doubled split-K chunk is of that size), that nothing outside the call's
own (tap, co, ci) entries changed, and that every gradient the user receives went through one checked call.

The fp64 reference of the filter gradient (`wgrad_reference`) is itself checked against torch autograd on the CPU."""
import ctypes
import inspect

import pytest
import torch
import torch.nn.functional as F

from artist_style_transfer_b200 import conv_geometry as cg


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference of ast_wgrad_gather (include/ast.h):
#   dw[u*s_u + v*s_v + co*s_co + ci*s_ci] += sum_{n, i<mi, j<mj} gout[n, oy0+so*i, ox0+so*j, co] * x[n, si*i+dy, si*j+dx, ci]
# for every launch and every tap t with taps[t] = (dy, dx), wtaps[t] = (u, v); coordinates out of range read 0.

def _window(t, y0, x0, sy, sx, mi, mj):
    """t[:, y0 + sy*i, x0 + sx*j, :] for i < mi, j < mj (any strides, any dtype), zero where the pixel is outside t."""
    _, h, w, _ = t.shape
    ys = y0 + sy * torch.arange(mi, device=t.device)
    xs = x0 + sx * torch.arange(mj, device=t.device)
    vy, vx = (ys >= 0) & (ys < h), (xs >= 0) & (xs < w)
    out = t.index_select(1, ys.clamp(0, h - 1)).index_select(2, xs.clamp(0, w - 1))
    out[:, ~vy] = 0
    out[:, :, ~vx] = 0
    return out


def wgrad_indices(launch, cout, cin, s_co, s_ci, s_u, s_v, device):
    """[ntaps, cout, cin] int64: the dw element each (tap, co, ci) of the launch accumulates into."""
    base = torch.tensor([u * s_u + v * s_v for u, v in launch.wtaps], dtype=torch.int64, device=device)
    co = torch.arange(cout, dtype=torch.int64, device=device) * s_co
    ci = torch.arange(cin, dtype=torch.int64, device=device) * s_ci
    return base[:, None, None] + co[None, :, None] + ci[None, None, :]


def _row_contribution(x64, g64, launch, n, i, ref_size, idx):
    """What grid row i of image n of `launch` adds to dw (all taps), as a flat fp64 vector of ref_size."""
    out = torch.zeros(ref_size, dtype=torch.float64, device=x64.device)
    g = _window(g64[n:n + 1], launch.oy0 + launch.so * i, launch.ox0, launch.so, launch.so, 1, launch.mj)[0, 0]
    for t, (dy, dx) in enumerate(launch.taps):
        xr = _window(x64[n:n + 1], launch.si * i + dy, dx, launch.si, launch.si, 1, launch.mj)[0, 0]
        out.index_add_(0, idx[t].flatten(), (g.t() @ xr).flatten())
    return out


def wgrad_reference(x, gout, launches, s_co, s_ci, s_u, s_v, reflect=False):
    """fp64 filter gradient of one `ops.wgrad_gather` call, computed on the tensors' own device.

    x: [N,H,W,Ci], gout: [N,Ho,Wo,Co] in logical NHWC order (any strides / dtype).  Returns flat fp64 vectors indexed like
    the call's dw (element offsets relative to dw's first element), of length max offset + 1:
      ref     the gradient;
      A       the same contraction of |gout| and |x|: the scale of the element-wise error bounds;
      mutant  ref without the contribution of ONE grid row of one image (the row whose contribution has the largest
              norm), i.e. what a kernel that lost one row's worth of pixels would produce;
    and `row` = (launch index, image, grid row) of that row."""
    assert not reflect, "no production call mirrors out-of-range coordinates in a filter gradient"
    x64, g64 = x.double(), gout.double()
    n, co, ci = x.shape[0], gout.shape[3], x.shape[3]
    idxs = [wgrad_indices(l, co, ci, s_co, s_ci, s_u, s_v, x.device) for l in launches]
    size = int(max(int(i.max()) for i in idxs)) + 1
    ref = torch.zeros(size, dtype=torch.float64, device=x.device)
    scale = torch.zeros_like(ref)
    best = (-1.0, None)
    for li, (l, idx) in enumerate(zip(launches, idxs)):
        g = _window(g64, l.oy0, l.ox0, l.so, l.so, l.mi, l.mj)                  # [N, mi, mj, Co]
        gt, ga = g.transpose(2, 3), g.abs()
        rowsq = torch.zeros(n, l.mi, dtype=torch.float64, device=x.device)
        for t, (dy, dx) in enumerate(l.taps):
            xt = _window(x64, dy, dx, l.si, l.si, l.mi, l.mj)                   # [N, mi, mj, Ci]
            per_row = torch.matmul(gt, xt)                                     # [N, mi, Co, Ci]: one product per grid row
            ref.index_add_(0, idx[t].flatten(), per_row.sum((0, 1)).flatten())
            scale.index_add_(0, idx[t].flatten(), torch.einsum("nijc,nijd->cd", ga, xt.abs()).flatten())
            rowsq += per_row.square().sum((2, 3))
            del per_row, xt
        v, k = rowsq.flatten().max(0)
        if float(v) > best[0]:
            best = (float(v), (li, int(k) // l.mi, int(k) % l.mi))
    li, img, row = best[1]
    mutant = ref - _row_contribution(x64, g64, launches[li], img, row, size, idxs[li])
    return ref, scale, mutant, best[1]


def _autograd_wgrad(fn, x, gy, wshape):
    w = torch.zeros(wshape, dtype=torch.float64, requires_grad=True)
    fn(x.permute(0, 3, 1, 2), w).backward(gy.permute(0, 3, 1, 2))
    return w.grad


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("k,s,pad,n,h,w,cin,cout", [(3, 1, 1, 2, 11, 9, 5, 7), (3, 2, 0, 2, 13, 11, 6, 4),
                                                    (3, 1, 0, 1, 7, 12, 3, 8)])
def test_reference_matches_autograd_conv(k, s, pad, n, h, w, cin, cout):
    """conv_fwd launches (stride 1 with zero padding read as out-of-range, stride 2 unpadded at odd sizes), dw in
    nn.Conv2d [cout][cin][k][k] order."""
    torch.manual_seed(k + s + h)
    launches = cg.conv_fwd(k, s, pad, h, w)
    x = torch.randn(n, h, w, cin, dtype=torch.float64)
    gy = torch.randn(n, launches[0].mi, launches[0].mj, cout, dtype=torch.float64)
    ref, scale, _, _ = wgrad_reference(x, gy, launches, cin * k * k, k * k, k, 1)
    want = _autograd_wgrad(lambda a, b: F.conv2d(a, b, stride=s, padding=pad), x, gy, (cout, cin, k, k))
    assert ref.shape == (want.numel(),)
    assert _rel(ref, want.flatten()) < 1e-13
    wa = _autograd_wgrad(lambda a, b: F.conv2d(a, b, stride=s, padding=pad), x.abs(), gy.abs(), (cout, cin, k, k))
    assert _rel(scale, wa.flatten()) < 1e-13


def test_reference_matches_autograd_conv_tap_major():
    """The tap-major [u][v][co][ci] strides that cnn.py passes for the 3x3 layers (stride-2 conv, reflect-padded input
    already materialised, like the transform net's buffers)."""
    torch.manual_seed(5)
    k, n, h, w, cin, cout = 3, 2, 15, 13, 8, 6
    launches = cg.conv_fwd(k, 2, 0, h, w)
    x = torch.randn(n, h, w, cin, dtype=torch.float64)
    gy = torch.randn(n, launches[0].mi, launches[0].mj, cout, dtype=torch.float64)
    ref, _, _, _ = wgrad_reference(x, gy, launches, cin, 1, k * cout * cin, cout * cin)
    want = _autograd_wgrad(lambda a, b: F.conv2d(a, b, stride=2), x, gy, (cout, cin, k, k))
    assert _rel(ref.view(k, k, cout, cin).permute(2, 3, 0, 1), want) < 1e-13


def test_reference_matches_autograd_conv_transpose_phases():
    """ConvTranspose2d(3, stride 2, padding 1, output_padding 1) as four phase launches (the last grid row of some phases
    reads row h_in of x, which is outside and reads 0); dw in nn.ConvTranspose2d [cin][cout][k][k] order."""
    torch.manual_seed(6)
    n, h, w, cin, cout = 2, 5, 7, 6, 4
    launches = cg.convT_fwd(3, 2, 1, 1, h, w)
    assert len(launches) == 4
    x = torch.randn(n, h, w, cin, dtype=torch.float64)
    gy = torch.randn(n, 2 * h, 2 * w, cout, dtype=torch.float64)
    ref, _, _, _ = wgrad_reference(x, gy, launches, 9, cout * 9, 3, 1)
    want = _autograd_wgrad(lambda a, b: F.conv_transpose2d(a, b, stride=2, padding=1, output_padding=1), x, gy,
                           (cin, cout, 3, 3))
    assert _rel(ref, want.flatten()) < 1e-13


@pytest.mark.parametrize("short", [0, 4])
def test_reference_matches_autograd_vertical_taps(short):
    """A 9-tap vertical launch (the row-folded 9x9 ends: dy = 0..8, dx = 0) against a (9, 1) kernel, dw in [dy][co][ci]
    order like the thin layers' gradient blocks; with `short` missing input rows the last grid rows read zeros."""
    torch.manual_seed(7 + short)
    n, mi, mj, cin, cout = 2, 12, 10, 5, 3
    launch = cg.Launch(mi, mj, 1, 1, 0, 0, [(d, 0) for d in range(9)], [(d, 0) for d in range(9)], 0)
    x = torch.randn(n, mi + 8 - short, mj, cin, dtype=torch.float64)
    gy = torch.randn(n, mi, mj, cout, dtype=torch.float64)
    ref, _, _, _ = wgrad_reference(x, gy, [launch], cin, 1, cout * cin, 0)
    want = _autograd_wgrad(lambda a, b: F.conv2d(F.pad(a, (0, 0, 0, short)), b), x, gy, (cout, cin, 9, 1))
    assert _rel(ref.view(9, cout, cin), want[..., 0].permute(2, 0, 1)) < 1e-13


def test_reference_mutant_is_one_grid_row_less():
    """The mutant equals the gradient of the same launches with that grid row of the output gradient set to zero."""
    torch.manual_seed(8)
    n, h, w, cin, cout = 3, 6, 5, 4, 5
    launches = cg.convT_fwd(3, 2, 1, 1, h, w)
    x = torch.randn(n, h, w, cin, dtype=torch.float64)
    gy = torch.randn(n, 2 * h, 2 * w, cout, dtype=torch.float64)
    gy[1] *= 3                                     # make image 1 carry the largest rows
    ref, _, mutant, (li, img, row) = wgrad_reference(x, gy, launches, 9, cout * 9, 3, 1)
    assert img == 1
    l = launches[li]
    gz = gy.clone()
    gz[img, l.oy0 + l.so * row, l.ox0::l.so][:l.mj] = 0
    want = _autograd_wgrad(lambda a, b: F.conv_transpose2d(a, b, stride=2, padding=1, output_padding=1), x, gz,
                           (cin, cout, 3, 3))
    assert _rel(mutant, want.flatten()) < 1e-13
    assert _rel(mutant, ref) > 1e-3


def decode_reduce_table(descs_dev, n_desc):
    """The ast_reduce_desc records of a device descriptor table (arena.reduce_table) as ctypes structs."""
    from artist_style_transfer_b200 import _lib
    arr = (_lib.ReduceDesc * n_desc)
    raw = descs_dev.cpu().numpy().tobytes()
    assert len(raw) == ctypes.sizeof(arr)
    return list(arr.from_buffer_copy(raw))


def test_reduce_table_decodes():
    from artist_style_transfer_b200 import _lib
    descs = (_lib.ReduceDesc * 2)()
    descs[0].src_off, descs[0].dst_off, descs[0].row_stride, descs[0].rows, descs[0].cols = 0, 40, 32, 4, 32
    descs[1].src_off, descs[1].dst_off, descs[1].row_stride, descs[1].rows, descs[1].cols = 1 << 33, 7, 3, 5, 3
    got = decode_reduce_table(_lib.device_bytes(descs, "cpu"), 2)
    assert [(d.src_off, d.dst_off, d.row_stride, d.rows, d.cols) for d in got] == [(0, 40, 32, 4, 32),
                                                                                   (1 << 33, 7, 3, 5, 3)]


# ---------------------------------------------------------------------------------------------------------------------
# The real calls of a real step.

# Filter gradients, element-wise: |got - ref| <= tau * A.  Strict mode (FFMA, fp32 operands): rounding of fp32 running
# sums, tau = 2^-16.  Fast mode (bf16 operands, tcgen05): the fp32 TMEM accumulator truncates at every accumulate step, a
# drift of about K/8 * 2^-25 of the sum over the K pixels of one CTA (DESIGN section 3); tau = 2^-13 covers K <= 32 K.
# Whole tensor: ||got - ref|| <= rtol * ||ref|| + eps * ||A||.
#   rtol: strict 1e-5.  Fast 2^-14: the thin kernels run 14.8 K (first layer) and 18.4 K (last layer) pixels per CTA at
#     B = 32, 256^2, where the truncation model gives 5.5e-5 / 6.9e-5 of a sum whose terms share a sign (measured 3.7e-5 on
#     the last layer); the other fast-mode launches stay below 1e-5.
#   eps: the rounding error of an fp32 sum is proportional to the partial sums, i.e. to A, not to |ref|.  The first
#     layer's output gradient comes from an InstanceNorm backward, whose per-image, per-channel spatial sum is zero, and
#     its input is the 0..255 image: its filter gradient is a small difference of large sums, ||A|| / ||ref|| ~ 10^2..10^3.
#     eps is the element-wise accuracy relative to A that the kernels reach on such sums (max err/A measured 7.5e-7 fast,
#     1.1e-7 strict on those layers), with margin: 2^-19 fast, 2^-22 strict.  Since ||got - ref|| <= max(err/A) * ||A||,
#     this term is what a cancelling sum needs and no more; a lost grid row still exceeds the bound (asserted per call).
WGRAD_TOL = {"fast": (2.0 ** -13, 2.0 ** -14, 2.0 ** -19), "fp32": (2.0 ** -16, 1e-5, 2.0 ** -22)}   # (tau, rtol, eps)
CHANNEL_SUM_TAU = 1e-5
BATCH_REDUCE_TAU = 1e-6
WGRAD_FAMILIES = ("wgrad_tc", "wgrad_thin", "wgrad_simt")


class _ArenaProbe:
    """Wraps ops.wgrad_gather / channel_sum / batch_reduce: snapshot the arena, record the family counters, run the real
    call once with unchanged arguments, synchronise, evaluate the fp64 reference and keep a record.  Asserts come after
    the step, so one failure reports every call."""

    def __init__(self, lib, ops, mode):
        self.lib, self.mode = lib, mode
        self.real = {name: getattr(ops, name) for name in ("wgrad_gather", "channel_sum", "batch_reduce")}
        self.gbuf = None
        self.wgrad, self.csum, self.bred = [], [], []

    def _base(self, t):
        base = t if t._base is None else t._base
        if self.gbuf is None:
            self.gbuf = base
        assert base is self.gbuf, "every gradient-arena writer must target the same arena"
        return base, (t.data_ptr() - base.data_ptr()) // base.element_size()

    def _call(self, name, args, kwargs):
        fam0 = self.lib.family_stats()
        out = self.real[name](*args, **kwargs)
        torch.cuda.synchronize()
        return out, self.lib.family_delta(fam0)

    @staticmethod
    def _changed_outside(before, after, inside):
        outside = torch.ones(before.numel(), dtype=torch.bool, device=before.device)
        outside[inside] = False
        return int((before.view(torch.int32)[outside] != after.view(torch.int32)[outside]).sum())

    def wgrad_gather(self, *args, **kwargs):
        a = inspect.signature(self.real["wgrad_gather"]).bind(*args, **kwargs)
        a.apply_defaults()
        a = a.arguments
        x, gout, launches, dw = a["x"], a["gout"], a["launches"], a["dw"]
        gbuf, off = self._base(dw)
        before = gbuf.clone()
        out, fam = self._call("wgrad_gather", args, kwargs)
        ref, scale, mutant, row = wgrad_reference(x, gout, launches, a["s_co"], a["s_ci"], a["s_u"], a["s_v"],
                                                  reflect=a["reflect"])
        idx = torch.cat([wgrad_indices(l, gout.shape[3], x.shape[3], a["s_co"], a["s_ci"], a["s_u"], a["s_v"],
                                       x.device).flatten() for l in launches])
        uniq = idx.unique()
        gidx = off + uniq
        got = gbuf[gidx].double() - before[gidx].double()
        r, sc, m = ref[uniq], scale[uniq], mutant[uniq]
        tau, rtol, eps = WGRAD_TOL[self.mode]
        err = (got - r).abs()
        a_norm = float(sc.norm())
        ratio = err / sc.clamp_min(1e-300)       # padding channels: A = 0, and the error must be 0 too
        fams = {f: fam[f][0] for f in WGRAD_FAMILIES if fam[f][0]}
        self.wgrad.append(dict(
            off=off, lo=int(gidx.min()), hi=int(gidx.max()), count=int(uniq.numel()), terms=int(idx.numel()),
            launches=len(launches), fams=fams,
            shapes=(tuple(x.shape), str(x.dtype)[6:], tuple(gout.shape), str(gout.dtype)[6:]),
            fro=_rel(got, r), fro_tol=rtol + eps * a_norm / float(r.norm()), kappa=a_norm / float(r.norm()),
            max_ratio=float(ratio.max()), bad=int((err > tau * sc).sum()), tau=tau,
            mutant=_rel(got, m), mutant_tol=rtol + eps * a_norm / float(m.norm()), row=row,
            changed_outside=self._changed_outside(before, gbuf, gidx)))
        return out

    def channel_sum(self, *args, **kwargs):
        a = inspect.signature(self.real["channel_sum"]).bind(*args, **kwargs).arguments
        x, dst = a["x"], a["out"]
        gbuf, off = self._base(dst)
        before = gbuf.clone()
        out, fam = self._call("channel_sum", args, kwargs)
        x64 = x.double()
        ref, scale = x64.sum((0, 1, 2)), x64.abs().sum((0, 1, 2))
        gidx = off + torch.arange(dst.numel(), device=dst.device)
        got = gbuf[gidx].double() - before[gidx].double()
        self.csum.append(dict(shape=tuple(x.shape), launches=fam["pointwise"][0], fro=_rel(got, ref),
                              max_ratio=float(((got - ref).abs() / scale).max()),
                              bad=int(((got - ref).abs() > CHANNEL_SUM_TAU * scale).sum()),
                              changed_outside=self._changed_outside(before, gbuf, gidx)))
        return out

    def batch_reduce(self, *args, **kwargs):
        a = inspect.signature(self.real["batch_reduce"]).bind(*args, **kwargs).arguments
        src, dst = a["src"], a["dst"]
        gbuf, off = self._base(dst)
        before = gbuf.clone()
        out, fam = self._call("batch_reduce", args, kwargs)
        refs, scales, gidx = [], [], []
        for d in decode_reduce_table(a["descs_dev"], a["n_desc"]):
            v = src.as_strided((d.rows, d.cols), (d.row_stride, 1), src.storage_offset() + d.src_off).double()
            refs.append(v.sum(0))
            scales.append(v.abs().sum(0))
            gidx.append(off + d.dst_off + torch.arange(d.cols, device=dst.device))
        ref, scale, gidx = torch.cat(refs), torch.cat(scales), torch.cat(gidx)
        assert gidx.unique().numel() == gidx.numel(), "two descriptors write the same gradient entry"
        got = gbuf[gidx].double()                   # the kernel stores (dst = sum), it does not accumulate
        self.bred.append(dict(n_desc=a["n_desc"], launches=fam["optim"][0], fro=_rel(got, ref),
                              max_ratio=float(((got - ref).abs() / scale.clamp_min(1e-300)).max()),
                              bad=int(((got - ref).abs() > BATCH_REDUCE_TAU * scale).sum()),
                              changed_outside=self._changed_outside(before, gbuf, gidx)))
        return out


@pytest.fixture(scope="module")
def ast():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import artist_style_transfer_b200 as m
    return m


def _build(ast, precision, seed=2):
    from oracle import weights
    net = ast.StyleTransfer(device=torch.device("cuda"), precision=precision)
    net.load_state_dict(weights.transfer_state_dict(seed), strict=True)
    vgg = ast.VGG16(vgg_path=None, precision=precision).cuda()
    vgg.load_state_dict(weights.vgg_state_dict(seed), strict=False)
    return net, vgg


WORKLOADS = [
    ("fast", 32, 256),     # the benchmark workload
    ("fast", 1, 1024),     # BASELINE config 5
    ("fp32", 4, 256),      # BASELINE config 1
    ("fp32", 1, 1024),     # config 5 in strict mode
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch,size", WORKLOADS, ids=[f"{m}-b{b}-{s}" for m, b, s in WORKLOADS])
def test_param_grad_launches_of_a_step(ast, monkeypatch, mode, batch, size):
    from artist_style_transfer_b200 import _lib, ops
    from oracle import weights
    net, vgg = _build(ast, mode)
    content = weights.content_batch(batch, size, 2).cuda()
    style = ast.style_grams_single(vgg, weights.style_image(size, 2).cuda(), batch)
    arena = net._arena_for(content.device)
    probe = _ArenaProbe(_lib, ops, mode)
    for name in probe.real:
        monkeypatch.setattr(ops, name, getattr(probe, name))
    fam0 = _lib.family_stats()
    ast.perceptual_step(net, vgg, content, style)        # eager: the probes synchronise, which graph capture forbids
    torch.cuda.synchronize()
    step = _lib.family_delta(fam0)
    monkeypatch.undo()

    stages, plans = arena.stages, arena.plans
    fails = []
    tag = f"{mode} B={batch} {size}^2"
    for rec in probe.wgrad:
        layer = [i for i, pl in enumerate(plans) if pl.g_off == rec["off"]]
        layer = layer[0] if layer else None
        fam = "/".join(f"{f}x{c}" for f, c in rec["fams"].items()) or "none"
        xs, xd, gs, gd = rec["shapes"]
        print(f"[{tag}] layer {layer} {fam}: x{xs} {xd}, gout{gs} {gd}: |err|/|ref| {rec['fro']:.2e} "
              f"(bound {rec['fro_tol']:.1e}, |A|/|ref| {rec['kappa']:.0f}), max err/A {rec['max_ratio']:.2e} "
              f"(tau {rec['tau']:.1e}), mutant {rec['mutant']:.2e} = {rec['mutant'] / rec['mutant_tol']:.1f}x its bound "
              f"(row {rec['row']})")
        where = f"layer {layer} ({fam})"
        if layer is None:
            fails.append(f"{where}: wrote at arena offset {rec['off']}, which is no filter-gradient region")
            continue
        last = layer == len(stages) - 1
        want = ("wgrad_thin" if layer == 0 or last else "wgrad_tc") if mode == "fast" else "wgrad_simt"
        if rec["fams"] != {want: rec["launches"]}:
            fails.append(f"{where}: expected {rec['launches']} {want} launches, counters say {rec['fams']}")
        if rec["fro"] > rec["fro_tol"]:
            fails.append(f"{where}: whole-tensor error {rec['fro']:.2e} > {rec['fro_tol']:.2e}")
        if rec["bad"]:
            fails.append(f"{where}: {rec['bad']} entries with |err| > tau*A (max err/A {rec['max_ratio']:.2e})")
        if not rec["mutant"] > rec["mutant_tol"]:
            fails.append(f"{where}: dropping grid row {rec['row']} changes the gradient by only {rec['mutant']:.2e}")
        if rec["changed_outside"]:
            fails.append(f"{where}: {rec['changed_outside']} arena entries outside its (tap, co, ci) set changed")
        if rec["terms"] != rec["count"]:
            fails.append(f"{where}: two (tap, co, ci) terms map to the same gradient entry")
    for rec in probe.csum:
        print(f"[{tag}] channel_sum x{rec['shape']}: |err|/|ref| {rec['fro']:.2e}, max err/A {rec['max_ratio']:.2e}")
        if rec["bad"] or rec["changed_outside"] or rec["launches"] != 1:
            fails.append(f"channel_sum: {rec}")
    for rec in probe.bred:
        print(f"[{tag}] batch_reduce {rec['n_desc']} columns sets: |err|/|ref| {rec['fro']:.2e}, "
              f"max err/A {rec['max_ratio']:.2e}")
        if rec["bad"] or rec["changed_outside"] or rec["launches"] != 1:
            fails.append(f"batch_reduce: {rec}")

    # completeness: every filter-gradient region written by exactly one checked call, covering it exactly
    for i, (st, pl) in enumerate(zip(stages, plans)):
        n_g = 1
        for d in pl.g_shape:
            n_g *= d
        hits = [r for r in probe.wgrad if r["lo"] < pl.g_off + n_g and r["hi"] >= pl.g_off]
        if len(hits) != 1 or (hits[0]["lo"], hits[0]["hi"], hits[0]["count"]) != (pl.g_off, pl.g_off + n_g - 1, n_g):
            fails.append(f"layer {i}: filter-gradient region [{pl.g_off}, {pl.g_off + n_g}) written by "
                         f"{[(r['lo'], r['hi'], r['count']) for r in hits]}")
    if len(probe.csum) != 1 or len(probe.bred) != 1:
        fails.append(f"channel_sum ran {len(probe.csum)} times, batch_reduce {len(probe.bred)} times")
    seen = sum(r["launches"] for r in probe.wgrad)
    total = sum(step[f][0] for f in WGRAD_FAMILIES)
    if seen != total:
        fails.append(f"the step ran {total} filter-gradient launches, the probes saw {seen}")
    assert not fails, "\n".join(fails)

    # what the user receives is exactly what was checked
    assert probe.gbuf is not None
    for p, view in zip(arena.params(), arena.grad_views(probe.gbuf)):
        assert p.grad is not None and torch.equal(p.grad, view)
    for st in stages:
        if st.norm:       # the conv bias in front of an InstanceNorm has no effect and no gradient
            assert bool((st.conv.bias.grad == 0).all())
