"""Thin Python wrappers over the C ABI (include/ast.h).  Tensors are passed in logical (N,H,W,C) order.

Everything here launches CUDA kernels from libast_b200.so on the current torch stream; nothing falls back
to PyTorch ops.
"""
import functools

import torch

from . import _lib
from . import conv_geometry as cg
from ._lib import CONV_REFLECT, CONV_RELU, CONV_TENSOR, GatherGeom, check, image, ptr, ref, stream_ptr

CONV_ROUND_TF32 = 8
TF32 = "tf32"   # pack_weights dtype: fp32 storage rounded to TF32

_DT = {torch.float32: _lib.AST_F32, torch.bfloat16: _lib.AST_BF16}

# ---- optional per-family CUDA-event timing (bench.py roofline leg); off by default, zero cost when off
_prof = None
PROFILE_DETAIL = False   # per-shape labels (scratch/layer_times.py)


class _timed:
    def __init__(self, label):
        self.label = label

    def __enter__(self):
        if _prof is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if _prof is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            _prof.append((self.label, self.e0, e1))
        return False


def profile_begin():
    global _prof
    _prof = []


def profile_end():
    """-> {label: (total_ms, launches)} measured with CUDA events on the launching stream."""
    global _prof
    torch.cuda.synchronize()
    out = {}
    for label, e0, e1 in _prof or []:
        ms, cnt = out.get(label, (0.0, 0))
        out[label] = (ms + e0.elapsed_time(e1), cnt + 1)
    _prof = None
    return out


def _geom(launch, flags=0, w_img_stride=0, stats=None, pooled=None, pool_codes=None):
    g = GatherGeom()
    g.mi, g.mj, g.si, g.so, g.oy0, g.ox0 = launch.mi, launch.mj, launch.si, launch.so, launch.oy0, launch.ox0
    g.ntaps = len(launch.taps)
    g.flags = flags
    for t, (dy, dx) in enumerate(launch.taps):
        g.dy[t] = dy
        g.dx[t] = dx
    g.w_img_stride = w_img_stride
    g.stats = None if stats is None else stats.data_ptr()
    if pooled is not None:
        g._pooled_img = pooled                      # keep the ctypes struct alive as long as the geometry
        g.pooled = _lib.ctypes.pointer(pooled)
    if pool_codes is not None:
        g._codes_img = pool_codes
        g.pool_codes = _lib.ctypes.pointer(pool_codes)
    return g


@functools.lru_cache(maxsize=None)
def _tap_offsets_cached(key, device_index):
    return torch.tensor(list(key), dtype=torch.int32, device=torch.device("cuda", device_index))


def tap_offsets(wtaps, s_u, s_v, device):
    """int32 device table of weight offsets u*s_u + v*s_v for each tap."""
    return _tap_offsets_cached(tuple(u * s_u + v * s_v for u, v in wtaps), device.index or 0)


def _pack_weights_impl(w, launches, a, b, s_a, s_b, s_u, s_v, dtype):
    """Pack fp32 master weights into [taps][a][b] (`dtype`) for the given launches (ast_pack_weights)."""
    wt = cg.all_wtaps(launches)
    offs = tap_offsets(wt, s_u, s_v, w.device)
    out = torch.empty((len(wt), a, b), dtype=torch.float32 if dtype == TF32 else dtype, device=w.device)
    code = 2 if dtype == TF32 else _DT[dtype]
    check(_lib.load().ast_pack_weights(ptr(w), ptr(offs), len(wt), a, b, s_a, s_b, ptr(out), code,
                                       stream_ptr()), "ast_pack_weights")
    return out


def _pw(name, t):
    return "pointwise" + (f"|{name}{tuple(t.shape)}" if PROFILE_DETAIL and _prof is not None else "")


def pack_weights_ex(w, tap_offs, a, a_valid, b, b_valid, b0, s_a, s_b1, s_b0, dtype):
    """dst[t][ia][ib] = w.flat[tap_offs[t] + ia*s_a + (ib//b0)*s_b1 + (ib%b0)*s_b0], zero outside the valid box."""
    with _timed("pack"):
        offs = _tap_offsets_cached(tuple(tap_offs), w.device.index or 0)
        out = torch.empty((len(tap_offs), a, b), dtype=torch.float32 if dtype == TF32 else dtype, device=w.device)
        code = 2 if dtype == TF32 else _DT[dtype]
        check(_lib.load().ast_pack_weights_ex(ptr(w), ptr(offs), len(tap_offs), a, a_valid, b, b_valid, b0, s_a, s_b1,
                                              s_b0, ptr(out), code, stream_ptr()), "ast_pack_weights_ex")
        return out


def row_im2col(src, out, kw, sign, px, py, reflect, shift=None, round_tf32=False):
    """out[n,y,x,d*C+c] = src[n, y-py, x+sign*d-px, c] (+shift); see include/ast.h ast_row_im2col."""
    with _timed(_pw("row_im2col", out)):
        si, oi = image(src), image(out)
        check(_lib.load().ast_row_im2col(ref(si), ref(oi), ptr(shift), kw, sign, px, py, int(reflect), int(round_tf32),
                                         stream_ptr()), "ast_row_im2col")
        return out


def _flip(img):
    """Channel-reversed alias of an ast_image (BGR <-> RGB, inference.py:116 `[[2, 1, 0]]`): same pixels, channel c of the
    view is channel C-1-c of the tensor - expressed with a negative channel stride, no kernel support needed."""
    esz = {_lib.AST_F32: 4, _lib.AST_BF16: 2, _lib.AST_U8: 1}[img.dtype]
    img.ptr = img.ptr + (img.c - 1) * img.sc * esz
    img.sc = -img.sc
    return img


def fold_rows(part, out, kw, bias=None, relu=False, flip_channels=False):
    """out[n,y,x,c] = bias[c] + sum_d part[n,y,x+d,d*C+c]; see include/ast.h ast_fold_rows."""
    with _timed(_pw("fold_rows", part)):
        pi, oi = image(part), image(out)
        if flip_channels:
            oi = _flip(oi)
        check(_lib.load().ast_fold_rows(ref(pi), ref(oi), ptr(bias), kw, int(relu), stream_ptr()), "ast_fold_rows")
        return out


def instnorm_finalize(sums, n, c, hw, eps=1e-5):
    """(sum x, sum x^2) pairs accumulated by a conv epilogue -> (mean, rstd)."""
    with _timed("instnorm"):
        mean = torch.empty(n * c, dtype=torch.float32, device=sums.device)
        rstd = torch.empty_like(mean)
        check(_lib.load().ast_instnorm_finalize(ptr(sums), n, c, hw, eps, ptr(mean), ptr(rstd), stream_ptr()),
              "ast_instnorm_finalize")
        return mean, rstd


def tc_eligible(x, cout):
    """Shapes the tcgen05 kernel accepts (conv_tc.cu): cin*elemsize % 64 == 0, cout % 32 == 0, NHWC."""
    return (_lib.has_tc_conv() and x.stride(3) == 1 and (x.shape[3] * x.element_size()) % 64 == 0
            and cout % 32 == 0 and cout in (32, 64, 128, 256, 512))


def _conv_gather_impl(x, wpacked, launches, out, bias=None, in_shift=None, add=None, mask=None, relu=False,
                reflect=False, tensor=False, w_img_stride=0, round_tf32=False, stats=None, pooled=None,
                pool_only=False, pool_codes=None):
    """Run every launch of an op. x/out/add/mask: (N,H,W,C)-ordered tensors; wpacked: [taps][cout][cin].
    pooled: optional (N,H/2,W/2,C) tensor receiving MaxPool2d(2,2) of the result (weight-stationary kernel only);
    pool_codes: optional uint8 (N,H/2,W/2,C) window codes for the pooling backward (include/ast.h)."""
    lib = _lib.load()
    flags = ((CONV_RELU if relu else 0) | (CONV_REFLECT if reflect else 0) | (CONV_TENSOR if tensor else 0)
             | (CONV_ROUND_TF32 if round_tf32 else 0) | (_lib.CONV_POOL_ONLY if pool_only else 0))
    xi, oi, ai, mi = image(x), image(out), image(add), image(mask)
    pooled = image(pooled)
    pool_codes = image(pool_codes)
    cout, cin = wpacked.shape[-2], wpacked.shape[-1]
    esz = wpacked.element_size()
    for l in launches:
        g = _geom(l, flags, w_img_stride, stats, pooled, pool_codes)
        wp = _lib.ctypes.c_void_p(wpacked.data_ptr() + l.woff * cout * cin * esz)
        check(lib.ast_conv_gather(ref(xi), wp, ptr(bias), ptr(in_shift), ref(ai), ref(mi), ref(oi), ref(g),
                                  stream_ptr()), "ast_conv_gather")
    return out


def _conv_stacked_impl(x, wstacked, stk, out, bias=None, add=None, mask=None, relu=False, round_tf32=False, stats=None):
    lib = _lib.load()
    g = _lib.StackedGeom()
    g.nblk, g.mi, g.mj, g.sy, g.soy, g.sox = stk.nblk, stk.mi, stk.mj, stk.sy, stk.soy, stk.sox
    for b in range(stk.nblk):
        g.oy[b], g.ox[b] = stk.oy[b], stk.ox[b]
    g.nvt, g.ntaps = len(stk.vt), stk.ntaps
    g.flags = (CONV_RELU if relu else 0) | (CONV_ROUND_TF32 if round_tf32 else 0)
    for v, (dy, dx) in enumerate(stk.vt):
        g.dy[v], g.dx[v] = dy, dx
    g.stats = stats.data_ptr() if stats is not None else None
    if wstacked.shape[0] != len(stk.vt) or wstacked.shape[1] != 128 or wstacked.shape[2] != x.shape[3] or wstacked.dtype != x.dtype:
        raise RuntimeError(f"conv_stacked: stacked filter {tuple(wstacked.shape)} {wstacked.dtype} does not match "
                           f"{len(stk.vt)} virtual taps x 128 x {x.shape[3]} {x.dtype}")
    xi, oi, ai, mi = image(x), image(out), image(add), image(mask)
    check(lib.ast_conv_stacked(ref(xi), ptr(wstacked), ptr(bias), ref(ai), ref(mi), ref(oi), ref(g), stream_ptr()),
          "ast_conv_stacked")
    return out


def conv_stacked(x, wstacked, stk, out, bias=None, add=None, mask=None, relu=False, round_tf32=False, stats=None):
    """Block-stacked tensor-core convolution for 32/64-channel outputs (include/ast.h ast_conv_stacked).
    stk: conv_geometry.Stacked; wstacked: [virtual taps][128][cin] (stack_filter / the arena's stacked packs)."""
    label = "conv_stacked"
    if PROFILE_DETAIL and _prof is not None:
        label += f"|{tuple(x.shape)}->{tuple(out.shape)} vt={len(stk.vt)} {str(x.dtype)[6:]}"
    with _timed(label):
        return _conv_stacked_impl(x, wstacked, stk, out, bias=bias, add=add, mask=mask, relu=relu, round_tf32=round_tf32,
                                  stats=stats)


def stack_filter(tile_of, stk, cb, cin, dtype, device):
    """[virtual taps][128][cin] stacked filter of a conv_geometry.Stacked launch; tile_of(kernel position) -> [cb][cin]
    operand tile ([cout][cin] orientation) of that filter tap.  One-time host-driven build (frozen VGG filters, tests); the
    TransformerNet's stacked filters are written by the fused optimizer kernel (arena.py)."""
    w = torch.zeros(len(stk.vt), 128, cin, dtype=dtype, device=device)
    for v, row in enumerate(stk.src):
        for g, pos in enumerate(row):
            if pos is not None:
                w[v, g * cb:(g + 1) * cb] = tile_of(pos).to(dtype)
    return w


def tc_contract_eligible(a, b):
    """Operands the tcgen05 contraction kernel accepts (contract_tc.cu): NHWC, same dtype, 16-byte pixel stride."""
    ok = _lib.has_tc_gram() and a.dtype == b.dtype
    for t in (a, b):
        ok = ok and t.stride(3) == 1 and all((s * t.element_size()) % 16 == 0 for s in t.stride()[:3])
    return ok


def _wgrad_gather_impl(x, gout, launches, dw, s_co, s_ci, s_u, s_v, reflect=False, tensor=False):
    """dw (fp32, pre-zeroed) += filter gradient for every launch of the op."""
    lib = _lib.load()
    flags = (CONV_REFLECT if reflect else 0) | (CONV_TENSOR if tensor else 0)
    xi, gi = image(x), image(gout)
    for l in launches:
        offs = tap_offsets(l.wtaps, s_u, s_v, dw.device)
        g = _geom(l, flags)
        check(lib.ast_wgrad_gather(ref(xi), ref(gi), ptr(dw), ptr(offs), s_co, s_ci, ref(g), stream_ptr()),
              "ast_wgrad_gather")
    return dw


_ws_cache = {}


def _workspace(nbytes, device):
    key = (device.index or 0)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def _instnorm_stats_impl(x, eps=1e-5):
    n, _, _, c = x.shape
    mean = torch.empty(n * c, dtype=torch.float32, device=x.device)
    rstd = torch.empty_like(mean)
    lib = _lib.load()
    ws = _workspace(lib.ast_instnorm_workspace_bytes(n, c), x.device)
    xi = image(x)
    check(lib.ast_instnorm_stats(ref(xi), ptr(mean), ptr(rstd), eps, ptr(ws), stream_ptr()), "ast_instnorm_stats")
    return mean, rstd


def _instnorm_apply_impl(x, mean, rstd, gamma, beta, out, pad, relu, residual=None):
    xi, oi, ri = image(x), image(out), image(residual)
    check(_lib.load().ast_instnorm_apply(ref(xi), ptr(mean), ptr(rstd), ptr(gamma), ptr(beta), ref(ri), ref(oi),
                                         pad, int(relu), stream_ptr()), "ast_instnorm_apply")
    return out


def _instnorm_bwd_impl(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal=None, s12=None, arrive=None):
    """Returns s12 of shape (2, N*C): dbeta = s12[0].view(N,C).sum(0), dgamma = s12[1].view(N,C).sum(0); fills dx
    (and gtotal).  `s12` may be a caller-provided (2, N*C) fp32 view (e.g. a slice of one buffer shared by layers) and
    `arrive` N int32 barrier counters; both must be zero-filled.  Zeroed buffers are allocated for those not given."""
    n, _, _, c = x.shape
    if s12 is None:
        s12 = torch.zeros((2, n * c), dtype=torch.float32, device=x.device)  # one allocation: the caller reduces both
    s1, s2 = s12[0], s12[1]                                                  # over the batch with one kernel
    if arrive is None:
        arrive = torch.zeros(n, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    xi, gp, ge, dxi, gt = image(x), image(gpad), image(gextra), image(dx), image(gtotal)
    check(lib.ast_instnorm_bwd(ref(xi), ptr(mean), ptr(rstd), ptr(gamma), ptr(beta), ref(gp), pad, ref(ge), int(relu),
                               ptr(s1), ptr(s2), ptr(arrive), ref(dxi), ref(gt), stream_ptr()), "ast_instnorm_bwd")
    return s12


def _maxpool2_fwd_impl(x, codes=None, out_dtype=None):
    n, h, w, c = x.shape
    y = torch.empty((n, h // 2, w // 2, c), dtype=out_dtype or x.dtype, device=x.device)
    xi, yi, ci = image(x), image(y), image(codes)
    check(_lib.load().ast_maxpool2_fwd(ref(xi), ref(yi), ref(ci), stream_ptr()), "ast_maxpool2_fwd")
    return y


def _maxpool2_bwd_impl(x, gy, gadd=None, codes=None):
    n, hp, wp, c = gy.shape
    shape = x.shape if x is not None else (n, 2 * hp, 2 * wp, c)
    gx = torch.empty(shape, dtype=gy.dtype, device=gy.device)
    xi, gyi, gai, gxi, ci = image(x if codes is None else None), image(gy), image(gadd), image(gx), image(codes)
    check(_lib.load().ast_maxpool2_bwd(ref(xi), ref(ci), ref(gyi), ref(gai), ref(gxi), stream_ptr()), "ast_maxpool2_bwd")
    return gx


def _gram_impl(x, scale, tensor=False):
    n, _, _, c = x.shape
    g = torch.empty((n, c, c), dtype=torch.float32, device=x.device)
    if n == 0 or c == 0:
        return g
    xi = image(x)
    check(_lib.load().ast_gram(ref(xi), ptr(g), scale, CONV_TENSOR if tensor else 0, stream_ptr()), "ast_gram")
    return g


def _mse_impl(a, b, loss, scale, grad=None, gscale=0.0):
    ai, bi, gi = image(a), image(b), image(grad)
    check(_lib.load().ast_mse(ref(ai), ref(bi), ptr(loss), scale, ref(gi), gscale, stream_ptr()), "ast_mse")
    return loss


def _copy_image_impl(src, dst, shift=None, pad=0, flip_channels=False):
    si, di = image(src), image(dst)
    if flip_channels:
        di = _flip(di)
    check(_lib.load().ast_copy_image(ref(si), ref(di), ptr(shift), pad, stream_ptr()), "ast_copy_image")
    return dst


def _accumulate_impl(x, acc):
    xi, ai = image(x), image(acc)
    check(_lib.load().ast_accumulate(ref(xi), ref(ai), stream_ptr()), "ast_accumulate")
    return acc


def _mask_add_impl(a, b, mask, out):
    ai, bi, mi, oi = image(a), image(b), image(mask), image(out)
    check(_lib.load().ast_mask_add(ref(ai), ref(bi), ref(mi), ref(oi), stream_ptr()), "ast_mask_add")
    return out


def pack_weights(w, launches, a, b, s_a, s_b, s_u, s_v, dtype):
    with _timed("pack"):
        return _pack_weights_impl(w, launches, a, b, s_a, s_b, s_u, s_v, dtype)


def conv_gather(x, wpacked, launches, out, bias=None, in_shift=None, add=None, mask=None, relu=False, reflect=False,
                tensor=False, w_img_stride=0, round_tf32=False, stats=None, pooled=None, pool_only=False, pool_codes=None):
    label = "conv_gather_tc" if tensor else "conv_gather_simt"
    if PROFILE_DETAIL and _prof is not None:
        label += f"|{tuple(x.shape)}->{tuple(out.shape)} taps={sum(len(l.taps) for l in launches)} {str(x.dtype)[6:]}"
    with _timed(label):
        return _conv_gather_impl(x, wpacked, launches, out, bias=bias, in_shift=in_shift, add=add, mask=mask, relu=relu,
                                 reflect=reflect, tensor=tensor, w_img_stride=w_img_stride, round_tf32=round_tf32,
                                 stats=stats, pooled=pooled, pool_only=pool_only, pool_codes=pool_codes)


def wgrad_gather(x, gout, launches, dw, s_co, s_ci, s_u, s_v, reflect=False, tensor=False):
    label = "wgrad_tc" if tensor else "wgrad_simt"
    if PROFILE_DETAIL and _prof is not None:
        label += f"|x{tuple(x.shape)} g{tuple(gout.shape)} taps={sum(len(l.taps) for l in launches)}"
    with _timed(label):
        return _wgrad_gather_impl(x, gout, launches, dw, s_co, s_ci, s_u, s_v, reflect=reflect, tensor=tensor)


def instnorm_stats(x, eps=1e-5):
    with _timed("instnorm" + (f"|stats{tuple(x.shape)}" if PROFILE_DETAIL and _prof is not None else "")):
        return _instnorm_stats_impl(x, eps=eps)


def instnorm_apply(x, mean, rstd, gamma, beta, out, pad, relu, residual=None):
    with _timed("instnorm" + (f"|apply{tuple(x.shape)}" if PROFILE_DETAIL and _prof is not None else "")):
        return _instnorm_apply_impl(x, mean, rstd, gamma, beta, out, pad, relu, residual=residual)


def instnorm_bwd(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal=None, s12=None, arrive=None):
    """`s12` and `arrive` (n int32 barrier counters), when given, are zero-filled by the caller: one fill for all layers."""
    with _timed("instnorm" + (f"|bwd{tuple(x.shape)}" if PROFILE_DETAIL and _prof is not None else "")):
        return _instnorm_bwd_impl(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal=gtotal, s12=s12,
                                  arrive=arrive)


def maxpool2_fwd(x, codes=None, out_dtype=None):
    """MaxPool2d(2,2); codes: optional uint8 (N,H/2,W/2,C) output with the window codes the backward can use instead of x.
    out_dtype: e.g. torch.float16 for a pooled tensor that only feeds the next fast-mode VGG convolution."""
    with _timed(_pw("maxpool_fwd", x)):
        return _maxpool2_fwd_impl(x, codes=codes, out_dtype=out_dtype)


def maxpool2_bwd(x, gy, gadd=None, codes=None):
    """gx = (route(gy) + gadd) * (x > 0); with `codes` (from the forward) x is not read (and may be None)."""
    with _timed(_pw("maxpool_bwd", gy)):
        return _maxpool2_bwd_impl(x, gy, gadd=gadd, codes=codes)


def gram(x, scale, tensor=False):
    with _timed("gram"):
        return _gram_impl(x, scale, tensor=tensor)


def gram_mse(x, target, g, counters, loss=None, loss_scale=0.0, d=None, d_scale=0.0, tensor=False):
    """Fused style term of one tap (include/ast.h ast_gram_mse): fills g = Gram(x) * 1/(CHW) (g and counters must be
    zero on entry), loss (an fp64 accumulator) += loss_scale * sum (g - target)^2, d = d_scale * (g - target).
    target: [C,C] (shared by the batch) or [N,C,C]."""
    if loss is not None and loss.dtype != torch.float64:
        raise RuntimeError("gram_mse: the loss accumulator must be float64")
    n, h, w, c = x.shape
    if n == 0 or c == 0:
        return g
    tstride = 0 if target.dim() == 2 or target.stride(0) == 0 else target.stride(0)
    if target.stride(-1) != 1 or target.stride(-2) != c:
        raise RuntimeError("gram_mse: target rows must be dense")
    with _timed("gram"):
        xi = image(x)
        check(_lib.load().ast_gram_mse(ref(xi), ptr(g), 1.0 / (c * h * w), ptr(target), tstride, ptr(loss), loss_scale,
                                       ptr(d), d_scale, ptr(counters), CONV_TENSOR if tensor else 0, stream_ptr()),
              "ast_gram_mse")
    return g


def channel_sum(x, out):
    """out[c] += sum_{n,h,w} x[n,h,w,c] (include/ast.h ast_channel_sum)."""
    with _timed(_pw("channel_sum", x)):
        xi = image(x)
        check(_lib.load().ast_channel_sum(ref(xi), ptr(out), stream_ptr()), "ast_channel_sum")
    return out


def batch_reduce(src, dst, descs_dev, n_desc, max_cols):
    """dst[dst_off + c] = sum_r src[src_off + r*row_stride + c] for a device table of descriptors (ast_batch_reduce)."""
    with _timed("pointwise"):
        check(_lib.load().ast_batch_reduce(ptr(src), ptr(dst), ptr(descs_dev), n_desc, max_cols, stream_ptr()),
              "ast_batch_reduce")
    return dst


def mse(a, b, loss, scale, grad=None, gscale=0.0):
    with _timed(_pw("mse", a)):
        return _mse_impl(a, b, loss, scale, grad=grad, gscale=gscale)


def copy_image(src, dst, shift=None, pad=0, flip_channels=False):
    with _timed(_pw("copy_image", dst)):
        return _copy_image_impl(src, dst, shift=shift, pad=pad, flip_channels=flip_channels)


def reflect_fold(gpad, out, pad, add=None):
    """out = adjoint of copy_image(..., pad) applied to gpad (+ add); see include/ast.h ast_reflect_fold."""
    with _timed(_pw("reflect_fold", out)):
        gi, ai, oi = image(gpad), image(add), image(out)
        check(_lib.load().ast_reflect_fold(ref(gi), ref(ai), ref(oi), pad, stream_ptr()), "ast_reflect_fold")
        return out


def accumulate(x, acc):
    with _timed(_pw("accumulate", x)):
        return _accumulate_impl(x, acc)


def mask_add(a, b, mask, out):
    with _timed(_pw("mask_add", a)):
        return _mask_add_impl(a, b, mask, out)
