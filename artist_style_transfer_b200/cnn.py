"""B200-native mirror of the reference transform network (`/root/reference/cnn.py`).

Same class names, constructor arguments, forward signatures and `state_dict` keys as the reference
(`StyleTransfer` cnn.py:10-49, `ConvLayer` :52-79, `ResidualLayer` :82-99, `DeconvLayer` :102-124), so
reference checkpoints load with `strict=True`.  Underneath, every layer is a sequence of calls into
libast_b200.so (hand-written sm_100a kernels); there is no PyTorch-op or CPU fallback.

Internal data flow (DESIGN.md): activations are NHWC; each stage is
    gather-conv (raw, pre-norm)  ->  InstanceNorm stats  ->  fused apply (+ReLU, +residual) that writes the
    next conv's reflection-padded input buffer directly.
The backward pass runs the same stages in reverse inside one autograd.Function.
"""
import math

import torch
import torch.nn as nn

from . import arena as arena_mod
from . import conv_geometry as cg
from . import ops

# precision modes (north_star): 'fp32' = strict, FFMA kernels, fp32 activations;
# 'fast' = bf16 activations/weights for the transform net on tcgen05 where the shape is supported.
_MODES = ("fp32", "fast")
_default_mode = "fp32"


def set_default_precision(mode):
    global _default_mode
    if mode not in _MODES:
        raise ValueError(f"precision must be one of {_MODES}")
    _default_mode = mode


def get_default_precision():
    return _default_mode


class _ConvParams(nn.Module):
    """Parameter holder laid out like nn.Conv2d / nn.ConvTranspose2d (weight, bias) with PyTorch's default init."""

    def __init__(self, weight_shape, fan_in, bias_size):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(weight_shape))
        self.bias = nn.Parameter(torch.empty(bias_size))
        bound = 1.0 / math.sqrt(fan_in)
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)   # == kaiming_uniform_(a=sqrt(5))
            self.bias.uniform_(-bound, bound)


class _NormParams(nn.Module):
    """Parameter holder of nn.InstanceNorm2d(affine=True): weight=1, bias=0, no running stats."""

    def __init__(self, channels):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(channels))
        self.bias = nn.Parameter(torch.zeros(channels))


class _Stage:
    __slots__ = ("kind", "cin", "cout", "k", "stride", "opad", "norm", "relu", "res_from", "conv", "normp")

    def __init__(self, kind, cin, cout, k, stride, opad, norm, relu, res_from, conv, normp):
        self.kind, self.cin, self.cout, self.k, self.stride, self.opad = kind, cin, cout, k, stride, opad
        self.norm, self.relu, self.res_from, self.conv, self.normp = norm, relu, res_from, conv, normp

    @property
    def in_pad(self):
        return self.k // 2 if (self.kind == "conv" and self.k > 1) else 0


def _interior(t, p):
    return t if p == 0 else t[:, p:t.shape[1] - p, p:t.shape[2] - p, :]


def _fwd_geometry(st, hin, win):
    if st.kind == "conv":
        ls = cg.conv_fwd(st.k, st.stride, 0, hin, win)
        return ls, ls[0].mi, ls[0].mj
    ho = cg.convT_out_size(hin, st.k, st.stride, st.k // 2, st.opad)
    wo = cg.convT_out_size(win, st.k, st.stride, st.k // 2, st.opad)
    return cg.convT_fwd(st.k, st.stride, st.k // 2, st.opad, hin, win), ho, wo


def _vtaps(k, sign=1):
    taps = [(sign * dy, 0) for dy in range(k)]
    return taps, [(dy, 0) for dy in range(k)]


def _conv_packed(x, pk, launches, out, **kw):
    """One conv through an arena pack: the block-stacked tensor-core kernel when the arena laid the filter out for it
    (32/64-channel outputs: ConvTranspose phases, stride-2 data gradients, the vertical-tap forms of the 9x9 ends)."""
    if pk.stacked is None:
        return ops.conv_gather(x, pk.tensor, launches, out, **kw)
    kw.pop("tensor", None)
    groups = arena_mod.stack_groups(launches, out.shape[3])
    if len(groups) != len(pk.stacked):
        raise RuntimeError("block-stacked conv: the launches of this image size do not match the packed filter")
    for g, ref, vb in zip(groups, pk.stacked, pk.vbase):
        if g.vt != ref.vt or g.src != ref.src:
            raise RuntimeError("block-stacked conv: the taps of this image size do not match the packed filter")
        ops.conv_stacked(x, pk.tensor[vb:vb + len(g.vt)], g, out, **kw)
    return out


class _StageFunction(torch.autograd.Function):
    """Forward/backward of a list of stages as ONE autograd node.

    x: [N,3,H,W] (or [N,H,W,3] with nhwc=True), fp32 or uint8 -> [N,3,H,W] fp32 (or uint8 RGB [N,H,W,3] with u8_out, the
    fused post-processing of inference.py:116).  Packed weights come from the owner's TransferArena (one re-pack launch
    when a parameter changed); gradients are accumulated in the arena's flat tap-major layout (arena.py).
    """

    @staticmethod
    def forward(ctx, x, arena, nhwc, u8_out, *params):
        stages, mode, adt = arena.stages, arena.mode, arena.adt
        x_shape, x_dtype = x.shape, x.dtype
        x = x.detach()
        if x.dtype not in (torch.float32, torch.uint8):
            x = x.to(torch.float32)
        xv = x if nhwc else x.permute(0, 2, 3, 1)          # logical (N, H, W, C) view, no copy
        n, h, w, _ = xv.shape
        dev = x.device
        train = any(ctx.needs_input_grad)
        arena.ensure_packs()
        pit = iter(params)
        P = []
        for st in stages:
            cw, cb = next(pit), next(pit)
            P.append((cw, cb, next(pit), next(pit)) if st.norm else (cw, cb, None, None))
        plans = arena.plans
        p0 = stages[0].in_pad
        thin_in = plans[0].thin_in
        if thin_in:     # row-im2col of the reflect-padded image: [N, H+2p, W, 32] (k*cin channels used)
            node = torch.empty((n, h + 2 * p0, w, 32), dtype=adt, device=dev)
            ops.row_im2col(xv, node, stages[0].k, 1, p0, p0, True)
        else:
            node = torch.empty((n, h + 2 * p0, w + 2 * p0, stages[0].cin), dtype=adt, device=dev)
            ops.copy_image(xv, node, pad=p0)
        nodes, node_pad, saved = [node], [p0], []
        out = None
        # (sum x, sum x^2) of every InstanceNorm layer, accumulated in fp64 by the conv epilogues: one fill for all layers
        zeros = torch.zeros(max(1, sum(2 * n * st.cout for st in stages if st.norm)), dtype=torch.float64, device=dev)
        zoff = 0
        last_use = {}                                   # node index -> last stage that reads it (inference frees the rest)
        for i, st in enumerate(stages):
            last_use[i] = i
            if st.res_from is not None:
                last_use[st.res_from + 1] = i
        for i, st in enumerate(stages):
            cw, cb, gam, bet = P[i]
            pl = plans[i]
            xin = nodes[i]
            last = i == len(stages) - 1
            if i == 0 and thin_in:
                taps, wt = _vtaps(st.k)
                launches, ho, wo = [cg.Launch(h, w, 1, 1, 0, 0, taps, wt, 0)], h, w
            else:
                launches, ho, wo = _fwd_geometry(st, xin.shape[1], xin.shape[2])
                arena.woff(pl.fwd, launches)
            wp = pl.fwd.tensor
            if not st.norm:
                assert last, "a stage without norm must be the last one"
                if u8_out:
                    out = torch.empty((n, ho, wo, st.cout), dtype=torch.uint8, device=dev)
                    outv = out
                else:
                    out = torch.empty((n, st.cout, ho, wo), dtype=torch.float32, device=dev)
                    outv = out.permute(0, 2, 3, 1)
                if pl.thin_out:
                    # k vertical taps on the tensor cores give, per pixel, the partial sums of all k horizontal taps
                    # as k*cout (27 of 32) channels; ast_fold_rows adds the k shifted partials and the bias
                    taps, wt = _vtaps(st.k)
                    part = torch.empty((n, ho, xin.shape[2], 32), dtype=torch.float32, device=dev)
                    _conv_packed(xin, pl.fwd, [cg.Launch(ho, xin.shape[2], 1, 1, 0, 0, taps, wt, 0)], part, tensor=True)
                    ops.fold_rows(part, outv, st.k, bias=cb.detach(), relu=st.relu, flip_channels=u8_out)
                    del part
                else:
                    tmp = outv
                    if u8_out:                     # strict mode: fp32 result, then the clip / RGB / uint8 copy
                        tmp = torch.empty((n, ho, wo, st.cout), dtype=torch.float32, device=dev)
                    ops.conv_gather(xin, wp, launches, tmp, bias=cb.detach(), relu=st.relu)
                    if u8_out:
                        ops.copy_image(tmp, outv, flip_channels=True)
                saved.append((launches, None, None, None))
            else:
                raw = torch.empty((n, ho, wo, st.cout), dtype=adt, device=dev)
                # conv bias is dead under InstanceNorm (SURVEY 8b) and is not added
                use_tc = mode == "fast" and (ops.tc_eligible(xin, st.cout) or pl.fwd.stacked is not None)
                if use_tc:                         # sum x / sum x^2 accumulated by the conv epilogue: no stats pass
                    sums = zeros[zoff:zoff + 2 * n * st.cout]
                    zoff += 2 * n * st.cout
                    _conv_packed(xin, pl.fwd, launches, raw, tensor=True, stats=sums)
                    mean, rstd = ops.instnorm_finalize(sums, n, st.cout, ho * wo)
                else:
                    ops.conv_gather(xin, wp, launches, raw)
                    mean, rstd = ops.instnorm_stats(raw)
                pn = 0 if last else stages[i + 1].in_pad
                post = torch.empty((n, ho + 2 * pn, wo + 2 * pn, st.cout), dtype=adt, device=dev)
                res = None
                if st.res_from is not None:
                    j = st.res_from + 1
                    res = _interior(nodes[j], node_pad[j])
                ops.instnorm_apply(raw, mean, rstd, gam.detach(), bet.detach(), post, pn, st.relu, residual=res)
                nodes.append(post)
                node_pad.append(pn)
                saved.append((launches, raw if train else None, mean, rstd))
                del raw
                if last:
                    out = torch.empty((n, st.cout, ho, wo), dtype=torch.float32, device=dev)
                    ops.copy_image(post, out.permute(0, 2, 3, 1))
            if not train:                          # inference: drop every buffer nobody reads any more
                for j in range(min(i + 1, len(nodes))):
                    if nodes[j] is not None and last_use.get(j, j) <= i:
                        nodes[j] = None
                xin = None
        if train:
            ctx.arena, ctx.P = arena, P
            ctx.x_shape, ctx.x_dtype, ctx.nhwc = x_shape, x_dtype, nhwc
            ctx.nodes, ctx.node_pad, ctx.saved = nodes, node_pad, saved
        return out

    @staticmethod
    def backward(ctx, gout):
        arena, P, nodes, node_pad, saved = ctx.arena, ctx.P, ctx.nodes, ctx.node_pad, ctx.saved
        stages, plans, mode = arena.stages, arena.plans, arena.mode
        want_gx = ctx.needs_input_grad[0]
        adt = nodes[0].dtype
        gdt = adt                                   # dtype of the gradients flowing between layers
        gout = gout.to(torch.float32)
        dev = gout.device
        L = len(stages)
        gpad = [None] * (L + 1)
        gextra = [None] * (L + 1)
        sink = arena.grad_sink
        gbuf = sink if sink is not None else arena.new_grad_buffer()     # zeroed: the kernels accumulate into it
        nb = gout.shape[0]
        # per-(n,c) InstanceNorm-backward sums of every layer in ONE zeroed buffer; dbeta / dgamma of all layers then come
        # out of one batched column reduction
        bank_off, total = [], 0
        for st in stages:
            if st.norm:
                bank_off.append(total)
                total += 2 * nb * st.cout
        n_norm = len(bank_off)
        # + nb int32 barrier counters per layer for the single-kernel backward (same zero fill, viewed as int32)
        banks = torch.zeros(max(total + n_norm * nb, 1), dtype=torch.float32, device=dev)
        arrive_all = banks[total:].view(torch.int32)
        bank_it = len(bank_off)
        for i in reversed(range(L)):
            st, pl = stages[i], plans[i]
            cw, cb, gam, bet = P[i]
            launches, raw, mean, rstd = saved[i]
            xin = nodes[i]
            n_g = 1
            for d in pl.g_shape:
                n_g *= d
            g_w = gbuf[pl.g_off:pl.g_off + n_g].view(pl.g_shape)
            if not st.norm:
                d_raw = gout.permute(0, 2, 3, 1)
                ops.channel_sum(d_raw, gbuf[pl.g_cb:pl.g_cb + st.cout])
                if pl.thin_out:   # Dr[n,y,x',dx*cout+co] = dOut[n,y,x'-dx,co]: shared by the wgrad and the dgrad
                    pk = st.k // 2
                    hb, wb = gout.shape[2], gout.shape[3]
                    d_raw = torch.empty((nb, hb, wb + 2 * pk, 32), dtype=adt, device=dev)
                    ops.row_im2col(gout.permute(0, 2, 3, 1), d_raw, st.k, -1, 0, 0, False)
            else:
                j = i + 1
                n, ho, wo, c = raw.shape
                if i == L - 1:
                    ge = torch.empty((n, ho, wo, c), dtype=gdt, device=dev)
                    ops.copy_image(gout.permute(0, 2, 3, 1), ge)
                    gextra[j] = ge
                d_raw = torch.empty_like(raw)
                gtotal = torch.empty(raw.shape, dtype=gdt, device=dev) if st.res_from is not None else None
                bank_it -= 1
                s12 = banks[bank_off[bank_it]:bank_off[bank_it] + 2 * n * c].view(2, n * c)
                ops.instnorm_bwd(raw, mean, rstd, gam.detach(), bet.detach(), gpad[j], node_pad[j],
                                 gextra[j], st.relu, d_raw, gtotal, s12=s12,
                                 arrive=arrive_all[bank_it * nb:(bank_it + 1) * nb])
                if gtotal is not None:
                    assert gextra[st.res_from + 1] is None
                    gextra[st.res_from + 1] = gtotal
                gpad[j] = gextra[j] = None           # free
            wtc = mode == "fast" and ops.tc_contract_eligible(xin, d_raw)
            if i == 0 and pl.thin_in:
                # k vertical taps handled as a tap group inside the contraction kernel (d_raw loaded once per stage):
                # g_w[dy][co][dx*cin+c] += sum_p dY[p][co] * Xr[p + dy rows][dx*cin+c]
                ops.wgrad_gather(xin, d_raw, launches, g_w, 32, 1, st.cout * 32, 0, tensor=wtc)
            elif pl.thin_out:
                # g_w[dy][dx*cout+co][c] += sum_{y,x'} Dr[y][x'][dx*cout+co] * xin[y+dy][x'][c]
                taps, wt = _vtaps(st.k)
                lw = [cg.Launch(d_raw.shape[1], d_raw.shape[2], 1, 1, 0, 0, taps, wt, 0)]
                ops.wgrad_gather(xin, d_raw, lw, g_w, st.cin, 1, 32 * st.cin, 0, tensor=True)
            else:
                # tap-major scratch g_w[u][v][co][ci]: ci contiguous, so the contraction epilogue reduces with 16-byte
                # vector atomics; the optimizer / p.grad read it through strides
                ops.wgrad_gather(xin, d_raw, launches, g_w, st.cin, 1, st.k * st.cout * st.cin, st.cout * st.cin,
                                 tensor=wtc)
            if i == 0 and not want_gx:
                continue
            # data gradient w.r.t. node i (stage 0: its pack is built now, outside the arena)
            pk = pl.dgrad if i > 0 else arena.stage0_dgrad()
            if i == 0 and pl.thin_in:
                # gradient w.r.t. the reflect-padded 3-channel image as a 32 -> 3 k x k conv of d_raw in the last layer's
                # thin-output form: k vertical taps into k*cin partial channels, then ast_fold_rows
                k, p = st.k, st.in_pad
                n, h, w = d_raw.shape[:3]
                taps, wt = arena_mod.thin_in_dgrad_taps(k)
                part = torch.empty((n, h + 2 * p, w + 2 * (k - 1), 32), dtype=torch.float32, device=dev)
                _conv_packed(d_raw, pk, [cg.Launch(h + 2 * p, w + 2 * (k - 1), 1, 1, 0, 0, taps, wt, 0)], part, tensor=True)
                g_in = torch.empty((n, h + 2 * p, w + 2 * p, st.cin), dtype=torch.float32, device=dev)
                ops.fold_rows(part, g_in, k)
                del part
            elif pl.thin_out:
                taps, wt = _vtaps(st.k, -1)
                dl = [cg.Launch(xin.shape[1], xin.shape[2], 1, 1, 0, 0, taps, wt, 0)]
                g_in = torch.empty(xin.shape, dtype=gdt, device=dev)
                _conv_packed(d_raw, pk, dl, g_in, tensor=True)
            else:
                if st.kind == "conv":
                    dl = cg.conv_dgrad(st.k, st.stride, 0, xin.shape[1], xin.shape[2])
                else:
                    dl = cg.convT_dgrad(st.k, st.stride, st.k // 2, d_raw.shape[1], d_raw.shape[2])
                arena.woff(pk, dl)
                g_in = torch.empty(xin.shape, dtype=gdt, device=dev)
                src = d_raw
                if src.dtype != adt or not src.is_contiguous():   # fp32 NCHW grad of the last conv feeding the dgrad
                    src = torch.empty(d_raw.shape, dtype=adt, device=dev)
                    ops.copy_image(d_raw, src)
                _conv_packed(src, pk, dl, g_in, tensor=mode == "fast" and ops.tc_eligible(src, st.cin))
            gpad[i] = g_in
        gx = None
        if want_gx:
            # adjoint of how the forward wrote the input into node 0, plus the skip gradient of a standalone
            # ResidualLayer (node 0's interior is also its residual)
            gx = torch.empty(ctx.x_shape, dtype=ctx.x_dtype if ctx.x_dtype == torch.bfloat16 else torch.float32,
                             device=dev)
            ops.reflect_fold(gpad[0], gx if ctx.nhwc else gx.permute(0, 2, 3, 1), node_pad[0], add=gextra[0])
            gx = gx.to(ctx.x_dtype)
        if bank_off:
            ops.batch_reduce(banks, gbuf, *arena.reduce_table(nb, bank_off))
        ctx.nodes = ctx.saved = None
        if sink is not None:                         # the trainer reads the arena directly (p.grad are views of it)
            return (gx,) + (None,) * (3 + len(arena.params()))
        return (gx, None, None, None, *arena.grad_views(gbuf))


class _Precision:
    precision = None  # None -> module default (set_default_precision)

    def _mode(self):
        return self.precision or _default_mode

    def _arena_for(self, device):
        """TransferArena of this module's stage list for the current precision / device (built on first use)."""
        mode = self._mode()
        key = (mode, str(device))
        cache = self.__dict__.setdefault("_arenas", {})
        if key not in cache:
            a = arena_mod.TransferArena(self._stage_list(), mode, device)
            a.grad_sink = None
            cache[key] = a
        return cache[key]

    def _run(self, x, nhwc=False, u8_out=False):
        if not x.is_cuda:
            raise RuntimeError("StyleTransfer kernels run on CUDA only (no CPU fallback); move the module and "
                               "input to a B200")
        arena = self._arena_for(x.device)
        return _StageFunction.apply(x, arena, nhwc, u8_out, *arena.params())


class ConvLayer(nn.Module, _Precision):
    """ReflectionPad(k//2) -> Conv2d(k, stride) -> InstanceNorm2d(affine) (cnn.py:52-79)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, norm="instance"):
        super().__init__()
        if norm not in ("instance", "None"):
            raise ValueError("only norm='instance' or 'None' is on the accelerated path (cnn.py:66-70 'batch' is unused)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.norm_type = kernel_size, stride, norm
        self.conv_layer = _ConvParams((out_channels, in_channels, kernel_size, kernel_size),
                                      in_channels * kernel_size * kernel_size, out_channels)
        if norm == "instance":
            self.norm_layer = _NormParams(out_channels)

    def _stage(self, relu=False, res_from=None):
        return _Stage("conv", self.in_channels, self.out_channels, self.kernel_size, self.stride, 0,
                      self.norm_type == "instance", relu, res_from, self.conv_layer,
                      getattr(self, "norm_layer", None))

    def _stage_list(self):
        return [self._stage()]

    def forward(self, x):
        return self._run(x)


class ResidualLayer(nn.Module, _Precision):
    """conv2(relu(conv1(x))) + x, no activation after the add (cnn.py:82-99)."""

    def __init__(self, channels=128, kernel_size=3):
        super().__init__()
        self.conv1 = ConvLayer(channels, channels, kernel_size, stride=1)
        self.relu = nn.ReLU()
        self.conv2 = ConvLayer(channels, channels, kernel_size, stride=1)

    def _stages(self, base):
        """`base` = index of the stage whose output is this block's input (-1 = the run's input)."""
        return [self.conv1._stage(relu=True), self.conv2._stage(relu=False, res_from=base)]

    def _stage_list(self):
        return self._stages(-1)

    def forward(self, x):
        return self._run(x)


class DeconvLayer(nn.Module, _Precision):
    """ConvTranspose2d(k, stride, padding=k//2, output_padding) -> InstanceNorm2d(affine) (cnn.py:102-124)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride, output_padding, norm="instance"):
        super().__init__()
        if norm != "instance":
            raise ValueError("only norm='instance' is on the accelerated path")
        if (kernel_size, stride, output_padding) not in ((1, 1, 0), (3, 2, 1)):
            raise ValueError("DeconvLayer supports (k,stride,output_padding) = (1,1,0) or (3,2,1) (cnn.py:33-37)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.output_padding, self.norm_type = kernel_size, stride, output_padding, norm
        self.conv_transpose = _ConvParams((in_channels, out_channels, kernel_size, kernel_size),
                                          out_channels * kernel_size * kernel_size, out_channels)
        self.norm_layer = _NormParams(out_channels)

    def _stage(self, relu=False):
        return _Stage("deconv", self.in_channels, self.out_channels, self.kernel_size, self.stride,
                      self.output_padding, True, relu, None, self.conv_transpose, self.norm_layer)

    def _stage_list(self):
        return [self._stage()]

    def forward(self, x):
        return self._run(x)


class StyleTransfer(nn.Module, _Precision):
    """Johnson-style image transform net with the reference's two extra 1x1 layers (cnn.py:10-49).

    `StyleTransfer(state_dict_filename=None, device=None, precision=None)`; master parameters stay fp32
    (the reference's `.double()` at cnn.py:43 is not reproduced: fp64 has no tensor-core path, see DESIGN.md).
    """

    def __init__(self, state_dict_filename=None, device=None, precision=None):
        if device is None:
            device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        super().__init__()
        self.precision = precision
        self.ConvBlock = nn.Sequential(
            ConvLayer(3, 32, 9, 1), nn.ReLU(),
            ConvLayer(32, 64, 3, 2), nn.ReLU(),
            ConvLayer(64, 128, 3, 2), nn.ReLU(),
            ConvLayer(128, 128, 1, 1), nn.ReLU())
        self.ResidualBlock = nn.Sequential(*[ResidualLayer(128, 3) for _ in range(5)])
        self.DeconvBlock = nn.Sequential(
            DeconvLayer(128, 128, 1, 1, 0), nn.ReLU(),
            DeconvLayer(128, 64, 3, 2, 1), nn.ReLU(),
            DeconvLayer(64, 32, 3, 2, 1), nn.ReLU(),
            ConvLayer(32, 3, 9, 1, norm="None"))
        if state_dict_filename is not None:
            self.load_state_dict(torch.load(state_dict_filename, map_location=device), strict=True)
        self.to(device)

    def _stages(self):
        stages = []
        for block in (self.ConvBlock, self.ResidualBlock, self.DeconvBlock):
            mods = list(block)
            for idx, m in enumerate(mods):
                nxt_relu = idx + 1 < len(mods) and isinstance(mods[idx + 1], nn.ReLU)
                if isinstance(m, (ConvLayer, DeconvLayer)):
                    stages.append(m._stage(relu=nxt_relu))
                elif isinstance(m, ResidualLayer):
                    stages += m._stages(len(stages) - 1)
        return stages

    def _stage_list(self):
        return self._stages()

    def forward(self, x):
        """x: [B,3,H,W] BGR 0-255, fp32 (cnn.py:45-49) or uint8 (values widened in the first layer's loader)."""
        return self._run(x)

    def stylize(self, images):
        """Inference with the pre/post-processing of inference.py:107-116 fused into the end layers:
        images uint8 [B,H,W,3] BGR (cv2 layout) -> uint8 [B,H,W,3] RGB, i.e. the reference's
        `net(x.transpose(2,0,1))[[2,1,0]].transpose(1,2,0).clip(0,255).astype('uint8')` per image."""
        if images.dtype != torch.uint8 or images.dim() != 4 or images.shape[3] != 3:
            raise ValueError("stylize() takes uint8 [B,H,W,3] images")
        with torch.no_grad():
            return self._run(images, nhwc=True, u8_out=True)


TransformerNet = StyleTransfer  # north_star's name for the same network (SURVEY D1)
