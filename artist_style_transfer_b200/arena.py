"""Flat buffers behind the TransformerNet parameters (SURVEY 8f-1; train_cnn.py:247-248,333-334,375).

For one stage list (the whole `StyleTransfer`, or a single layer module used on its own) this object owns

  * the PACK arena: the bf16 / fp32 operand copies of every conv weight in the `[tap][cout][cin]` layouts the gather
    kernels read (forward and data-gradient orientation; the 3-channel ends in their row-folded layouts), refreshed by ONE
    table-driven launch (`ast_adam_step(update=0)`) whenever a parameter changed - instead of one pack launch per layer
    and pass;
  * the layout of the GRADIENT arena: one flat fp32 buffer in which every filter gradient sits in the tap-major layout
    the contraction kernels accumulate into, followed by the bias / gamma / beta gradients.  `PerceptualTrainer` zeroes
    it with one fill, lets the backward pass write into it, all-reduces it as it is (NCCL, one call, no flatten /
    unflatten copies) and hands it to the fused Adam kernel, which reads it through per-tensor index maps;
  * the Adam state (exp_avg, exp_avg_sq, device-resident lr / step) and the descriptor tables of `ast_adam_step`.

The nn.Parameters themselves are NOT moved: the kernels address them relative to the lowest parameter address.
"""
import ctypes

import torch

from . import _lib
from . import conv_geometry as cg
from ._lib import AdamState, PackMap, ParamDesc, ReduceDesc  # noqa: F401

_ALIGN_PACK = 256      # bytes: packed tensors are TMA sources (16-byte minimum), keep them on separate L2 lines
_DT_CODE = {torch.float32: _lib.AST_F32, torch.bfloat16: _lib.AST_BF16}


def _canonical_fwd(st):
    if st.kind == "conv":
        return cg.conv_fwd(st.k, st.stride, 0, 16 + st.k, 16 + st.k)
    return cg.convT_fwd(st.k, st.stride, st.k // 2, st.opad, 8, 8)


def _canonical_dgrad(st):
    if st.kind == "conv":
        return cg.conv_dgrad(st.k, st.stride, 0, 16 + st.k, 16 + st.k)
    return cg.convT_dgrad(st.k, st.stride, st.k // 2, 16, 16)


def stack_groups(launches, cb):
    """The block-stacked launches (conv_geometry.Stacked) that replace `launches` for a cb-channel output: the
    interleaved-row form of a single stride-1 launch, or the sub-pixel phases 128/cb at a time."""
    nb = 128 // cb
    if len(launches) == 1:
        return [cg.stack_rows(launches[0], nb)]
    assert len(launches) % nb == 0
    return [cg.stack_phases(launches[i:i + nb]) for i in range(0, len(launches), nb)]


def _stacked_pack(groups, cb, kdim, dtype, uv, pos_of, within, stride):
    """_Pack of the stacked filters [sum of virtual taps][128][kdim] of `groups`.  pos_of(u, v): the kernel position under
    which conv_geometry lists master tap (u, v); within(u, v): extra element offset inside its [cb][kdim] tile."""
    vbase, nv = [], 0
    for g in groups:
        vbase.append(nv)
        nv += len(g.vt)
    where = {}
    for gi, g in enumerate(groups):
        for pos, lst in g.places().items():
            where.setdefault(pos, []).extend(((vbase[gi] + v) * 128 + b * cb) * kdim for v, b in lst)
    taps, rep, rep_stride = [], None, 0
    for u, v in uv:
        offs = sorted(where[pos_of(u, v)])
        r = len(offs)
        d = offs[1] - offs[0] if r > 1 else 0
        assert all(offs[i + 1] - offs[i] == d for i in range(r - 1)), "copies of a tap must be equally spaced"
        assert rep in (None, r) and (r == 1 or rep is None or rep_stride == d)
        rep, rep_stride = r, d
        taps.append(offs[0] + within(u, v))
    pk = _Pack((nv, 128, kdim), dtype, taps, stride, None, rep, rep_stride, groups)
    pk.vbase = vbase
    return pk


class _Pack:
    """One packed copy: byte offset in the arena, shape, dtype and the element map of the master weight."""
    __slots__ = ("off", "shape", "dtype", "taps", "stride", "tapidx", "tensor", "rep", "rep_stride", "stacked", "vbase")

    def __init__(self, shape, dtype, taps, stride, tapidx=None, rep=1, rep_stride=0, stacked=None):
        self.shape, self.dtype, self.taps, self.stride, self.tapidx = shape, dtype, taps, stride, tapidx
        self.rep, self.rep_stride = rep, rep_stride      # copies of every element (row-interleaved stacked filters)
        self.stacked = stacked                           # [conv_geometry.Stacked] of the canonical launches, or None
        self.vbase = None                                # first virtual tap of each stacked group in the filter
        self.off, self.tensor = 0, None

    def nbytes(self):
        n = 1
        for d in self.shape:
            n *= d
        return n * (2 if self.dtype == torch.bfloat16 else 4)


class _StagePlan:
    __slots__ = ("thin_in", "thin_out", "fwd", "dgrad", "g_shape", "g_taps", "g_stride", "g_off", "g_cb", "g_gam", "g_bet")


def thin_in_dgrad_taps(k):
    """(taps, wtaps) of the data gradient of a thin-input stage, w.r.t. its reflect-padded cin-channel image P:
    part[n, Y, x, d*cin + c] = sum_{u, co} dY[n, Y - u, x - (k-1), co] * W[co, c, u, k-1-d] over a (h+2p, w+2(k-1)) grid,
    and ast_fold_rows then gives gP[n, Y, X, c] = sum_d part[n, Y, X + d, d*cin + c]."""
    return [(-u, -(k - 1)) for u in range(k)], [(u, 0) for u in range(k)]


def dgrad_pack(st, pl, tc, adt):
    """Layout of the data-gradient operand copy of one stage's filter.  The arena holds it for every stage but the first;
    TransferArena.stage0_dgrad builds the first stage's from the same layout when an input gradient is asked for."""
    k, co, ci = st.k, st.cout, st.cin
    conv = st.kind == "conv"
    uv = [(u, v) for u in range(k) for v in range(k)]
    if pl.thin_in:        # [u][d*cin + c][co] (k, 32, cout): a thin-output conv of dY, see thin_in_dgrad_taps
        taps, wt = thin_in_dgrad_taps(k)
        if (co * 2) % 128 == 0 or co * 2 == 64:
            vt = [cg.Launch(16, 16, 1, 1, 0, 0, taps, wt, 0)]
            return _stacked_pack(stack_groups(vt, 32), 32, co, adt, uv, lambda u, v: (u, 0),
                                 lambda u, v: (k - 1 - v) * ci * co, (1, co))
        return _Pack((k, 32, co), adt, [u * 32 * co + (k - 1 - v) * ci * co for u, v in uv], (1, co))
    if pl.thin_out:       # [dy][c][dx*cout + co] (k, cin, 32)
        if ci == 32:      # block-stacked: rows y - dy of the row-im2col'd output gradient
            vt_dg = [cg.Launch(16, 16, 1, 1, 0, 0, [(-u, 0) for u in range(k)], [(u, 0) for u in range(k)], 0)]
            return _stacked_pack(stack_groups(vt_dg, ci), ci, 32, adt, uv, lambda u, v: (u, 0), lambda u, v: v * co,
                                 (1, 32))
        return _Pack((k, ci, 32), adt, [u * ci * 32 + v * co for u, v in uv], (1, 32))
    # [t][ci][co], t in the order of the data-gradient launches' taps (phases for stride 2)
    canon = _canonical_dgrad(st)
    dg_stride = (1, co) if conv else (co, 1)
    if tc and conv and st.stride == 2 and ci in (32, 64) and (co * 2) % 128 == 0:
        # data gradient of a stride-2 conv: the 4 output phases as lane blocks
        return _stacked_pack(stack_groups(canon, ci), ci, co, adt, uv, lambda u, v: (u, v), lambda u, v: 0, dg_stride)
    order = cg.all_wtaps(canon)
    tapidx = {t: n for n, t in enumerate(order)}
    return _Pack((k * k, ci, co), adt, [tapidx[t] * ci * co for t in uv], dg_stride, tapidx)


def _param_desc(p_off, s_off, dims, g_off, g_stride, g_tap, packs, add_taps):
    """ast_param_desc of one parameter tensor; add_taps(list) -> first index of `list` in the tap table."""
    d = ParamDesc()
    d.p_off, d.s_off = p_off, s_off
    numel = 1
    for n_, v in enumerate(dims):
        d.dim[n_] = v
        numel *= v
    d.numel = numel
    d.g_off, d.g_tap, d.n_pack = g_off, g_tap, len(packs)
    d.g_stride[0], d.g_stride[1] = g_stride
    for n_, pk in enumerate(packs):
        d.pack[n_].off, d.pack[n_].tap, d.pack[n_].dtype = pk.off, add_taps(pk.taps), _DT_CODE[pk.dtype]
        d.pack[n_].stride[0], d.pack[n_].stride[1] = pk.stride
        d.pack[n_].rep, d.pack[n_].rep_stride = pk.rep, pk.rep_stride
    return d


class TransferArena:
    def __init__(self, stages, mode, device, thin_in_ok=True):
        self.stages, self.mode, self.device = list(stages), mode, device
        self.adt = torch.bfloat16 if mode == "fast" else torch.float32
        tc = mode == "fast" and _lib.has_tc_conv()
        self.tc = tc
        self.plans = []
        goff = 0

        def take(n):
            nonlocal goff
            o = goff
            goff += (n + 3) // 4 * 4            # 16-byte aligned segments (vector atomics, float4 reads)
            return o

        for i, st in enumerate(self.stages):
            pl = _StagePlan()
            k, k2, co, ci = st.k, st.k * st.k, st.cout, st.cin
            conv = st.kind == "conv"
            pl.thin_in = bool(tc and thin_in_ok and i == 0 and conv and st.stride == 1 and k > 1 and ci * k <= 32
                              and co % 32 == 0 and st.norm)
            pl.thin_out = bool(tc and i == len(self.stages) - 1 and conv and st.stride == 1 and k > 1 and co * k <= 32
                               and ci % 32 == 0 and not st.norm)
            uv = [(u, v) for u in range(k) for v in range(k)]
            sa_sb = (ci, 1) if conv else (1, ci)          # element (a, b) of the master weight -> [co][ci] position
            vt_fwd = [cg.Launch(16, 16, 1, 1, 0, 0, [(u, 0) for u in range(k)], [(u, 0) for u in range(k)], 0)]
            if pl.thin_in:        # [dy][co][dx*cin + c] (k, cout, 32): the row-im2col'd first layer, k vertical taps
                if co == 32:      # block-stacked (ast_conv_stacked): 4 interleaved output rows share every MMA
                    pl.fwd = _stacked_pack(stack_groups(vt_fwd, co), co, 32, self.adt, uv, lambda u, v: (u, 0),
                                           lambda u, v: v * ci, (32, 1))
                else:
                    pl.fwd = _Pack((k, co, 32), self.adt, [u * co * 32 + v * ci for u, v in uv], (32, 1))
                pl.g_shape, pl.g_taps, pl.g_stride = (k, co, 32), [u * co * 32 + v * ci for u, v in uv], (32, 1)
            elif pl.thin_out:     # [dy][dx*cout + co][c] (k, 32, cin): k vertical taps producing k*cout partial channels
                if (ci * 2) % 128 == 0 or ci * 2 == 64:
                    pl.fwd = _stacked_pack(stack_groups(vt_fwd, 32), 32, ci, self.adt, uv, lambda u, v: (u, 0),
                                           lambda u, v: v * co * ci, (ci, 1))
                else:
                    pl.fwd = _Pack((k, 32, ci), self.adt, [u * 32 * ci + v * co * ci for u, v in uv], (ci, 1))
                pl.g_shape, pl.g_taps, pl.g_stride = (k, 32, ci), [u * 32 * ci + v * co * ci for u, v in uv], (ci, 1)
            else:                 # [t][co][ci], t in the order of the forward launches' taps
                canon = _canonical_fwd(st)
                if tc and not conv and st.stride == 2 and co in (32, 64) and (ci * 2) % 128 == 0:
                    # ConvTranspose2d stride 2: the 4 sub-pixel phases as lane blocks of one (cout 32) / two (cout 64) launches
                    pl.fwd = _stacked_pack(stack_groups(canon, co), co, ci, self.adt, uv, lambda u, v: (u, v),
                                           lambda u, v: 0, sa_sb)
                else:
                    order = cg.all_wtaps(canon)
                    tapidx = {t: n for n, t in enumerate(order)}
                    pl.fwd = _Pack((k2, co, ci), self.adt, [tapidx[t] * co * ci for t in uv], sa_sb, tapidx)
                # tap-major gradient scratch [u][v][co][ci]: ci contiguous -> 16-byte vector reductions in the epilogue
                pl.g_shape, pl.g_taps, pl.g_stride = (k, k, co, ci), [(u * k + v) * co * ci for u, v in uv], sa_sb
            # the first stage's input gradient is optional: its pack is built on demand (stage0_dgrad)
            pl.dgrad = dgrad_pack(st, pl, tc, self.adt) if i > 0 else None
            n = 1
            for d in pl.g_shape:
                n *= d
            pl.g_off = take(n)
            pl.g_cb = take(co)
            pl.g_gam = take(co) if st.norm else None
            pl.g_bet = take(co) if st.norm else None
            self.plans.append(pl)
        self.g_numel = goff
        # ---- pack arena
        poff = 0
        for pl in self.plans:
            for pk in (pl.fwd, pl.dgrad):
                if pk is not None:
                    pk.off = poff
                    poff += (pk.nbytes() + _ALIGN_PACK - 1) // _ALIGN_PACK * _ALIGN_PACK
        self.pack_arena = torch.zeros(max(poff, _ALIGN_PACK), dtype=torch.uint8, device=device)
        for pl in self.plans:
            for pk in (pl.fwd, pl.dgrad):
                if pk is not None:
                    pk.tensor = self.pack_arena[pk.off:pk.off + pk.nbytes()].view(pk.dtype).view(pk.shape)
        self._tables_key = None
        self._packs_key = None
        self.opt = None            # Adam state once enable_optimizer() was called
        self._reduce_cache = {}
        self._dg0_tables = None    # (weight address, descriptor, work list, work items, tap table) of stage0_dgrad

    # ------------------------------------------------------------------ parameters
    def params(self):
        out = []
        for st in self.stages:
            out += [st.conv.weight, st.conv.bias]
            if st.norm:
                out += [st.normp.weight, st.normp.bias]
        return out

    def _build_tables(self):
        """Descriptor / work / tap tables of ast_adam_step for the CURRENT parameter addresses."""
        params = self.params()
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("TransformerNet master parameters must be contiguous fp32 tensors")
            _lib._check_device(p)
        base = min(p.data_ptr() for p in params)
        taps = [0]
        descs, work = [], []
        item = _lib.load().ast_adam_work_item()
        s_off = 0

        def add_taps(lst):
            o = len(taps)
            taps.extend(int(x) for x in lst)
            return o

        def add_desc(p, dims, g_off, g_stride, g_tap, packs):
            nonlocal s_off
            assert (p.data_ptr() - base) % 4 == 0
            idx = len(descs)
            descs.append(_param_desc((p.data_ptr() - base) // 4, s_off, dims, g_off, g_stride, g_tap, packs, add_taps))
            for start in range(0, p.numel(), item):
                work.append((idx, start))
            s_off += (p.numel() + 3) // 4 * 4

        for st, pl in zip(self.stages, self.plans):
            w = st.conv.weight
            add_desc(w, tuple(w.shape), pl.g_off, pl.g_stride, add_taps(pl.g_taps),
                     [pk for pk in (pl.fwd, pl.dgrad) if pk is not None])
            add_desc(st.conv.bias, (st.cout, 1, 1, 1), pl.g_cb, (1, 0), 0, [])
            if st.norm:
                add_desc(st.normp.weight, (st.cout, 1, 1, 1), pl.g_gam, (1, 0), 0, [])
                add_desc(st.normp.bias, (st.cout, 1, 1, 1), pl.g_bet, (1, 0), 0, [])
        self.n_desc, self.n_work, self.state_numel = len(descs), len(work), s_off
        self.descs_dev = _lib.device_bytes((ParamDesc * len(descs))(*descs), self.device)
        flat = (ctypes.c_int32 * (2 * len(work)))(*[x for pair in work for x in pair])
        self.work_dev = _lib.device_bytes(flat, self.device)
        self.taps_dev = torch.tensor(taps, dtype=torch.int64, device=self.device)
        self.base_ptr = base

    def _ptr_key(self):
        return tuple(p.data_ptr() for p in self.params())

    def _tables(self):
        key = self._ptr_key()
        if key != self._tables_key:
            if self.opt is not None and self._tables_key is not None:
                raise RuntimeError("TransformerNet parameters were re-allocated (e.g. .to()/.float()) after the fused "
                                   "optimizer was created; build the PerceptualTrainer after moving the module")
            self._build_tables()
            self._tables_key = key
            self._packs_key = None

    # ------------------------------------------------------------------ packs
    def ensure_packs(self):
        """Re-pack (one launch) if any parameter changed since the packs were last written."""
        self._tables()
        key = tuple(p._version for p in self.params())
        if key != self._packs_key:
            self._launch(update=False, gbuf=None)
            self._packs_key = key

    def _launch(self, update, gbuf):
        lib = _lib.load()
        vp = ctypes.c_void_p
        o = self.opt
        _lib.check(lib.ast_adam_step(vp(self.descs_dev.data_ptr()), self.n_desc, vp(self.work_dev.data_ptr()), self.n_work,
                                     vp(self.base_ptr), _lib.ptr(gbuf), _lib.ptr(o["m"]) if update else None,
                                     _lib.ptr(o["v"]) if update else None, vp(self.pack_arena.data_ptr()),
                                     vp(self.taps_dev.data_ptr()), _lib.ptr(o["state"]) if update else None,
                                     1 if update else 0, _lib.stream_ptr()), "ast_adam_step")

    def stage0_dgrad(self):
        """The first stage's data-gradient filter (dgrad_pack layout, outside the pack arena), written from the current
        weights by one ast_adam_step(update=0) launch over a one-descriptor table: the arena's packing code, stacked
        replicas included.  Written on every call, never cached: the fused Adam updates the parameters in place without
        bumping their versions, and a CUDA graph that captures the backward must capture this launch with it.  Only the
        device tables are kept (they depend on the weight's address, not its values)."""
        st, pl = self.stages[0], self.plans[0]
        w = st.conv.weight
        pk = dgrad_pack(st, pl, self.tc, self.adt)
        t = self._dg0_tables
        if t is None or t[0] != w.data_ptr():
            if w.dtype != torch.float32 or not w.is_contiguous():
                raise RuntimeError("TransformerNet master parameters must be contiguous fp32 tensors")
            taps = []

            def add_taps(lst):
                taps.extend(int(x) for x in lst)
                return 0
            d = _param_desc(0, 0, tuple(w.shape), 0, (0, 0), 0, [pk], add_taps)
            item = _lib.load().ast_adam_work_item()
            work = [x for s in range(0, w.numel(), item) for x in (0, s)]
            t = (w.data_ptr(), _lib.device_bytes(d, self.device),
                 _lib.device_bytes((ctypes.c_int32 * len(work))(*work), self.device), len(work) // 2,
                 torch.tensor(taps, dtype=torch.int64, device=self.device))
            self._dg0_tables = t
        buf = torch.zeros(pk.nbytes(), dtype=torch.uint8, device=self.device)   # zero rows of the stacked layouts
        vp = ctypes.c_void_p
        _lib.check(_lib.load().ast_adam_step(vp(t[1].data_ptr()), 1, vp(t[2].data_ptr()), t[3], _lib.ptr(w), None, None,
                                             None, vp(buf.data_ptr()), vp(t[4].data_ptr()), None, 0, _lib.stream_ptr()),
                   "ast_adam_step")
        pk.tensor = buf.view(pk.dtype).view(pk.shape)
        return pk

    def woff(self, pack, launches):
        """Rewrite each launch's first-tap index for the canonical tap order of `pack` (robust to skipped phases)."""
        if pack.tapidx is not None:
            for l in launches:
                l.woff = pack.tapidx[l.wtaps[0]]
        return launches

    # ------------------------------------------------------------------ gradients
    def new_grad_buffer(self):
        return torch.zeros(self.g_numel, dtype=torch.float32, device=self.device)

    def grad_views(self, gbuf):
        """Per-parameter views of the gradient arena shaped like the parameters (strided for conv weights)."""
        out = []
        for st, pl in zip(self.stages, self.plans):
            k = st.k
            su, sv = pl.g_taps[k] if k > 1 else 0, pl.g_taps[1] if k > 1 else 0
            sa, sb = pl.g_stride
            out.append(gbuf.as_strided(tuple(st.conv.weight.shape), (sa, sb, su, sv), pl.g_off))
            out.append(gbuf[pl.g_cb:pl.g_cb + st.cout])
            if st.norm:
                out.append(gbuf[pl.g_gam:pl.g_gam + st.cout])
                out.append(gbuf[pl.g_bet:pl.g_bet + st.cout])
        return out

    def reduce_table(self, n, bank_offsets):
        """Device descriptors of ast_batch_reduce: dbeta / dgamma of every InstanceNorm layer from its (2, n, c) sums."""
        key = (n, tuple(bank_offsets))
        hit = self._reduce_cache.get(key)
        if hit is None:
            descs, maxc = [], 0
            it = iter(bank_offsets)
            for st, pl in zip(self.stages, self.plans):
                if not st.norm:
                    continue
                off = next(it)
                for which, dst in ((0, pl.g_bet), (1, pl.g_gam)):
                    d = ReduceDesc()
                    d.src_off, d.dst_off, d.row_stride = off + which * n * st.cout, dst, st.cout
                    d.rows, d.cols = n, st.cout
                    descs.append(d)
                maxc = max(maxc, st.cout)
            hit = (_lib.device_bytes((ReduceDesc * len(descs))(*descs), self.device), len(descs), maxc)
            self._reduce_cache[key] = hit
        return hit

    # ------------------------------------------------------------------ optimizer
    def enable_optimizer(self, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4):
        self._tables()
        st = AdamState()
        st.lr, st.beta1, st.beta2, st.eps, st.weight_decay, st.grad_scale = lr, betas[0], betas[1], eps, weight_decay, 1.0
        st.step, st.bias_c1, st.bias_c2 = 0.0, 1.0, 1.0
        self.opt = {"m": torch.zeros(self.state_numel, dtype=torch.float32, device=self.device),
                    "v": torch.zeros(self.state_numel, dtype=torch.float32, device=self.device),
                    "state": _lib.device_bytes(st, self.device).view(torch.float32)}

    def set_lr(self, lr):
        self.opt["state"][0:1].fill_(float(lr))          # device scalar: the captured graph reads it at replay time

    def adam_step(self, gbuf):
        self._tables()
        self._launch(update=True, gbuf=gbuf)
        # the kernel refreshed the packs from the updated parameters; parameter versions did not change
        self._packs_key = tuple(p._version for p in self.params())
