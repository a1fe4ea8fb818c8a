"""Every InstanceNorm launch of a training step and of `stylize`, against fp64 of its own operands.

The InstanceNorm family (`csrc/norm.cu`) is the largest non-convolution cost of the step: `ast_instnorm_finalize` turns
the sums fused into a tensor-core conv epilogue into mean / rstd, `ast_instnorm_stats` computes them from the conv
output in strict mode, `ast_instnorm_apply` writes the next conv's reflect-padded input (+ReLU, +residual), and
`ast_instnorm_bwd` runs the backward of pad o ReLU o (+residual) o InstanceNorm in one cooperative launch or two.  The
staged kernels split rows into segments, images into row blocks and pick one or two launches by an L2 / co-residency
rule; the step-level parity tests cannot see a launch that is wrong at one segment seam or one border pixel.

Here a real `perceptual_step` (and a 1080p `stylize`) runs with the four entry points wrapped.  Each call fills its
outputs with NaN, runs once with unchanged arguments and is compared with fp64 of exactly the operands it received; it
must write every element of its outputs, change nothing else in their storage (for the backward: the rest of the shared
sums buffer), leave its inputs bit-identical and run the launches its plan promises.  The backward's sum bounds come from
the plan (`ns_plan_py`, a restatement of `ns_plan` that the barrier counters validate).  Each call must also fail
against the mutants that apply to it.  The fp64 references are held to torch autograd on the CPU."""
import inspect
import time

import pytest
import torch
import torch.nn.functional as F

from test_conv_launch_kernels import WORKLOADS, _bits, _changed_outside, _inside, _site, _storage_view
from test_param_grad_kernels import _build

U = 2.0 ** -24                 # fp32 unit roundoff
OUT_ROUND = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8}
# Element bounds (|err| <= tau * sum of the magnitudes the kernel's fp32 arithmetic adds + the store's rounding):
#   apply: A = gamma*rstd, A*mean, D = beta - A*mean, fma(A, x, D), + res: <= 5 roundings of a partial <= the scale;
#   g' (fold of up to 9 padded positions + gextra, pad 4 at H = 5): <= 10 roundings;
#   dx = A*g' + B*x + C with B, C folded from four fp32 products each, on top of g': <= 16 roundings.
APPLY_TAU = 8 * U
GPRIME_TAU = 16 * U
DX_TAU = 32 * U
NS_CONSUMERS, NS_SLAB_MAX, NS_SMEM_BUDGET, NS_MAX_STAGES = 256, 16384, 100 * 1024, 8
STATS_THREADS = 256
# DESIGN section 5: InstanceNorm launches of one step at B = 32, 256^2, fast mode
STEP_B32 = dict(in_apply=17, bwd_single=13, bwd_double=4)
IN_FAMILIES = ("in_apply", "in_bwd", "in_stats")


def gamma_k(k):
    """Higham's bound on the relative error of a recursive fp32 sum of depth k (relative to the sum of |terms|)."""
    return k * U / (1 - k * U)


# ---------------------------------------------------------------------------------------------------------------------
# The launch plans of csrc/norm.cu, restated.

def ns_plan_py(n, c, h, w, pad, rows_total, width, esz, nslabs, sms, slab_max=NS_SLAB_MAX, budget=NS_SMEM_BUDGET):
    """ns_plan: segments of the iterated row, ring stages, row blocks per image; None when the shape cannot be staged."""
    extra = 2 * pad if width != w else 0
    seg_max = slab_max // (c * esz) - extra
    if seg_max < 4 * pad + 1:
        return None
    nseg = -(-width // seg_max)
    seg = -(-width // nseg)
    nseg = -(-width // seg)
    slab_bytes = -(-(seg + extra) * c * esz // 128) * 128
    stages = min(budget // (nslabs * slab_bytes), NS_MAX_STAGES)
    if stages < 2:
        return None
    nblk = max(1, min(2 * sms // n, rows_total))
    return dict(nblk=nblk, seg=seg, nseg=nseg, stages=stages, slab_bytes=slab_bytes, rows=rows_total, width=width,
                slots=NS_CONSUMERS // (c // (16 // esz)))


def bwd_plan(n, c, h, w, pad, esz, nslabs, sms):
    """ast_instnorm_bwd: one cooperative launch when x + g' stay in L2 and every block is resident, else two."""
    scratch = 2 * (NS_CONSUMERS // (c // (16 // esz))) * c * 4
    if nslabs * n * h * w * c * esz <= 104e6:
        p = ns_plan_py(n, c, h, w, pad, h, w, esz, nslabs, sms, 8192 if nslabs == 3 else NS_SLAB_MAX,
                       NS_SMEM_BUDGET + 8192 - scratch)
        if p and p["nblk"] * n <= 2 * sms and p["stages"] * nslabs * p["slab_bytes"] + scratch + 128 <= 110 * 1024:
            return dict(p, launches=1)
    p = ns_plan_py(n, c, h, w, pad, h, w, esz, nslabs, sms)
    return None if p is None else dict(p, launches=2)


def bwd_depth(p):
    """Longest chain of fp32 additions behind one s1 / s2 entry: the pixels of one consumer thread, the block's slots,
    the blocks' atomics."""
    ppt = -(-p["rows"] // p["nblk"]) * p["nseg"] * -(-p["seg"] // p["slots"])
    return ppt + p["slots"] + p["nblk"]


def stats_plan(n, c, h, w, esz, sms):
    """ast_instnorm_stats: per-thread shifted sums over `chunk` pixels of `nblk` blocks, Chan merges over slots and blocks."""
    slots = STATS_THREADS // (c // (16 // esz))
    hw = h * w
    nblk = max(1, min(-(-4 * sms // n), -(-hw // (slots * 4))))
    chunk = -(-hw // nblk)
    return dict(nblk=nblk, slots=slots, depth=-(-chunk // slots) + slots + nblk)


# ---------------------------------------------------------------------------------------------------------------------
# fp64 references (NHWC, on the tensors' own device).

def reflect_index(n_out, pad, n, device):
    i = (torch.arange(n_out, device=device) - pad).abs()
    return torch.where(i >= n, 2 * (n - 1) - i, i)


def reflect_pad(t, pad):
    _, h, w, _ = t.shape
    return t[:, reflect_index(h + 2 * pad, pad, h, t.device)][:, :, reflect_index(w + 2 * pad, pad, w, t.device)]


def reflect_fold(gp, pad, h, w):
    """Adjoint of reflect_pad: [n, h+2p, w+2p, c] -> [n, h, w, c]."""
    n, _, wp, c = gp.shape
    t = torch.zeros((n, h, wp, c), dtype=gp.dtype, device=gp.device).index_add_(1, reflect_index(h + 2 * pad, pad, h, gp.device), gp)
    return torch.zeros((n, h, w, c), dtype=gp.dtype, device=gp.device).index_add_(2, reflect_index(wp, pad, w, gp.device), t)


def _per_image(v, n, c):
    return v.double().view(n, 1, 1, c)


def finalize_reference(sums, n, c, hw, eps=1e-5):
    """mean / rstd from (sum x, sum x^2) in fp64 and the bound of one fp32 rounding (+ fp64 noise of E[x^2] - mean^2)."""
    s = sums.double().view(n * c, 2)
    m = s[:, 0] / hw
    var = (s[:, 1] / hw - m * m).clamp_min(0)
    r = 1 / (var + eps).sqrt()
    dvar = 2.0 ** -50 * (s[:, 1].abs() / hw + m * m)
    return m, r, (U + 2.0 ** -50) * m.abs(), (U + 2.0 ** -50) * r + 0.51 * r * dvar / (var + eps)


def stats_reference(x, eps=1e-5):
    x64 = x.double()
    m = x64.mean((1, 2))
    var = (x64 - m[:, None, None]).square().mean((1, 2))
    return m.flatten(), (1 / (var + eps).sqrt()).flatten(), var.sqrt().flatten()


def apply_reference(x, mean, rstd, gamma, beta, pad, relu, res=None):
    """out = reflect_pad(ReLU(gamma*rstd*(x - mean) + beta (+ res))) from the call's own fp32 statistics, and the scale
    |A*x| + |A*mean| + |beta| (+ |res|) of the kernel's fp32 arithmetic (D = beta - A*mean cancels inside it)."""
    n, _, _, c = x.shape
    m, r = _per_image(mean, n, c), _per_image(rstd, n, c)
    A = gamma.double() * r
    x64 = x.double()
    y = A * (x64 - m) + beta.double()
    scale = (A * x64).abs() + (A * m).abs() + beta.double().abs()
    if res is not None:
        y = y + res.double()
        scale = scale + res.double().abs()
    if relu:
        y = y.clamp_min(0)
    return reflect_pad(y, pad), reflect_pad(scale, pad)


def bwd_sums(gp, xhat):
    return gp.sum((1, 2)).flatten(), (gp * xhat).sum((1, 2)).flatten()


def bwd_dx(gp, xhat, A, s1, s2, n, c, hw):
    return A * (gp - (s1.view(n, 1, 1, c) + xhat * s2.view(n, 1, 1, c)) / hw)


def bwd_reference(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu):
    """fp64 backward of pad o ReLU o (+res) o InstanceNorm with the call's fp32 mean / rstd: g' = (fold(gpad) + gextra) *
    [A*x + D > 0], s1 = sum g', s2 = sum g' * xhat, dx = A * (g' - (s1 + xhat * s2) / hw).  The mask is evaluated as the
    kernel does, on fp32 A and D; `amb` marks the pixels whose sign depends on whether D was rounded once (fma) or twice."""
    n, h, w, c = x.shape
    dev = x.device
    m, r = _per_image(mean, n, c), _per_image(rstd, n, c)
    A = gamma.double() * r
    x64 = x.double()
    xhat = (x64 - m) * r
    g = torch.zeros_like(x64)
    ga = torch.zeros_like(x64)
    if gpad is not None:
        gp64 = gpad.double()
        g, ga = reflect_fold(gp64, pad, h, w), reflect_fold(gp64.abs(), pad, h, w)
    if gextra is not None:
        g, ga = g + gextra.double(), ga + gextra.double().abs()
    if relu:
        a32 = (gamma.float().view(1, c) * rstd.view(n, c)).double()
        d_fma = (beta.double().view(1, c) - a32 * mean.double().view(n, c)).float().double()
        d_sep = (beta.float().view(1, c) - (a32.float() * mean.view(n, c))).double()
        a32, d_fma, d_sep = (t.view(n, 1, 1, c) for t in (a32, d_fma, d_sep))
        mask = (a32 * x64 + d_fma) > 0
        amb = mask != ((a32 * x64 + d_sep) > 0)
    else:
        mask = torch.ones(x.shape, dtype=torch.bool, device=dev)
        amb = torch.zeros(x.shape, dtype=torch.bool, device=dev)
    gp = g * mask
    s1, s2 = bwd_sums(gp, xhat)
    return dict(A=A, xhat=xhat, g=g, ga=ga * mask, gamb=g.abs() * amb, mask=mask, gp=gp, s1=s1, s2=s2,
                dx=bwd_dx(gp, xhat, A, s1, s2, n, c, h * w), amb=int(amb.sum()))


# ---------------------------------------------------------------------------------------------------------------------
# CPU checks of the references.

def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("pad,relu,res,gextra,h,w", [(1, True, False, False, 6, 7), (4, True, False, True, 5, 5),
                                                     (0, False, True, True, 4, 6), (2, False, True, False, 3, 9)])
def test_reference_apply_and_backward_match_autograd(pad, relu, res, gextra, h, w):
    """apply_reference = F.pad(reflect) o ReLU o (+res) o F.instance_norm, and bwd_reference's g', s1 = dbeta,
    s2 = dgamma (per image) and dx = autograd of the same composition, with gextra the gradient of a skip path that reads
    the post-ReLU output (h = pad + 1: every pixel on the border).  A forward residual only comes without a ReLU, as in
    the network's residual blocks: the backward's mask is A*x + D > 0."""
    torch.manual_seed(pad * 10 + h)
    n, c = 2, 5
    x = torch.randn(n, h, w, c, dtype=torch.float64) * 2 + 0.7
    gamma, beta = torch.rand(c, dtype=torch.float64) + 0.5, torch.randn(c, dtype=torch.float64)
    r = torch.randn(n, h, w, c, dtype=torch.float64) if res else None
    mean = x.mean((1, 2)).flatten()
    rstd = 1 / (x.var((1, 2), unbiased=False) + 1e-5).sqrt().flatten()
    gpad = torch.randn(n, c, h + 2 * pad, w + 2 * pad, dtype=torch.float64)
    ge = torch.randn(n, c, h, w, dtype=torch.float64) if gextra else None

    def head(pre):
        post = F.relu(pre) if relu else pre
        out = F.pad(post, (pad,) * 4, mode="reflect") if pad else post
        return out, (out * gpad).sum() + ((post * ge).sum() if gextra else 0)
    xa = _nchw(x).clone().requires_grad_(True)
    ga, ba = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    pre = F.instance_norm(xa, weight=ga, bias=ba, eps=1e-5) + (_nchw(r) if res else 0)
    out, loss = head(pre)
    got, scale = apply_reference(x, mean, rstd, gamma, beta, pad, relu, r)
    assert _rel(got, _nhwc(out.detach())) < 1e-13
    assert bool((scale >= got.abs() - 1e-12).all())
    loss.backward()
    ref = bwd_reference(x, mean, rstd, gamma, beta, _nhwc(gpad), pad, None if ge is None else _nhwc(ge), relu)
    assert _rel(ref["dx"], _nhwc(xa.grad)) < 1e-10
    assert _rel(ref["s1"].view(n, c).sum(0), ba.grad) < 1e-12
    assert _rel(ref["s2"].view(n, c).sum(0), ga.grad) < 1e-12
    pd = pre.detach().clone().requires_grad_(True)       # g' = the gradient at the ReLU's input
    head(pd)[1].backward()
    assert _rel(ref["gp"], _nhwc(pd.grad)) < 1e-13
    if not res:
        assert ref["amb"] == 0


def test_reference_fold_is_the_adjoint_of_reflect_pad():
    torch.manual_seed(3)
    for pad, h, w in ((1, 2, 3), (4, 5, 5), (3, 7, 4)):
        t = torch.randn(2, h, w, 3, dtype=torch.float64, requires_grad=True)
        g = torch.randn(2, h + 2 * pad, w + 2 * pad, 3, dtype=torch.float64)
        (F.pad(_nchw(t), (pad,) * 4, mode="reflect") * _nchw(g)).sum().backward()
        assert torch.allclose(reflect_fold(g, pad, h, w), t.grad, rtol=0, atol=1e-13)
        assert torch.equal(reflect_pad(t.detach(), pad), _nhwc(F.pad(_nchw(t.detach()), (pad,) * 4, mode="reflect")))


def test_reference_statistics():
    torch.manual_seed(4)
    x = torch.randn(3, 7, 9, 4, dtype=torch.float64) * 0.01 + 5
    m, r, _ = stats_reference(x)
    want = F.instance_norm(_nchw(x), eps=1e-5)
    assert _rel(_nhwc(want), (x - m.view(3, 1, 1, 4)) * r.view(3, 1, 1, 4)) < 1e-10
    s = torch.stack([x.sum((1, 2)), x.square().sum((1, 2))], -1).flatten()
    fm, fr, bm, br = finalize_reference(s, 3, 4, 63)
    assert _rel(fm, m) < 1e-15 and _rel(fr, r) < 1e-9
    assert bool((bm > 0).all() and (br > 0).all())


def test_plan_restatement():
    """ns_plan_py at the shapes the issue of segments and blocks is about (148 SMs): the 1928-column stylize apply runs 8
    segments, the seg_max edge (C=32 bf16 pad 1: 254 padded columns in one segment, 255 in two), n = 300 two launches."""
    assert ns_plan_py(1, 32, 1080, 1920, 4, 1088, 1928, 2, 1, 148)["nseg"] == 8
    assert ns_plan_py(2, 32, 9, 252, 1, 11, 254, 2, 1, 148)["nseg"] == 1
    assert ns_plan_py(2, 32, 9, 253, 1, 11, 255, 2, 1, 148)["nseg"] == 2
    assert ns_plan_py(2, 1024, 8, 8, 4, 16, 16, 2, 1, 148) is None
    assert bwd_plan(300, 32, 8, 8, 1, 2, 2, 148)["launches"] == 2
    assert bwd_plan(4, 128, 225, 225, 1, 2, 2, 148)["launches"] == 1
    assert bwd_plan(4, 128, 226, 226, 1, 2, 2, 148)["launches"] == 2
    p = bwd_plan(2, 128, 16, 70, 1, 2, 3, 148)
    assert p["launches"] == 1 and p["nseg"] == 3 and 70 - 2 * p["seg"] < p["seg"]
    assert bwd_plan(32, 32, 256, 256, 4, 2, 2, 148)["launches"] == 2


# ---------------------------------------------------------------------------------------------------------------------
# Checks of one call (shared by the probe and the standalone cases).

def _ratio(err, bound):
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def check_finalize(sums, n, c, hw, mean, rstd, eps=1e-5, row=None):
    m, r, bm, br = finalize_reference(sums, n, c, hw, eps)
    em, er = (mean.double() - m).abs(), (rstd.double() - r).abs()
    rec = dict(bad=int((em > bm).sum() + (er > br).sum()), ratio=max(_ratio(em, bm), _ratio(er, br)), mutants={})
    if row:
        mm, rm, _, _ = finalize_reference(sums, n, c, hw - row, eps)
        rec["mutants"]["hw_short"] = max(_ratio((mean.double() - mm).abs(), bm), _ratio((rstd.double() - rm).abs(), br))
    return rec


def check_stats(x, mean, rstd, sms, eps=1e-5):
    """mean and rstd of strict-mode statistics against fp64: |d mean| <= gamma_k * (|mean| + std) and |d rstd| / rstd <=
    gamma_k * (2 + 2 |mean| / std), k = pixels per thread + slots + blocks (the Chan merges: a mean off by d shifts M2 by
    at most 2 d * hw * std)."""
    n, h, w, c = x.shape
    p = stats_plan(n, c, h, w, x.element_size(), sms)
    m, r, sd = stats_reference(x, eps)
    gk = gamma_k(p["depth"] + 4)
    bm = gk * (m.abs() + sd)
    br = gk * (2 + 2 * m.abs() / sd.clamp_min(1e-300)) * r
    em, er = (mean.double() - m).abs(), (rstd.double() - r).abs()
    return dict(bad=int((em > bm).sum() + (er > br).sum()), ratio=max(_ratio(em, bm), _ratio(er, br)), mutants={},
                plan=p, mu_sd=float((m.abs() / sd.clamp_min(1e-300)).max()), rel_rstd=float((er / r).max()))


def check_apply(x, mean, rstd, gamma, beta, res, out, pad, relu, sms):
    """out against apply_reference, element-wise within APPLY_TAU * scale + the store's rounding, every element written;
    mutants: zero padding, no residual, the last image with another image's statistics, one row of the last image with
    the first column of segment 1 taken from the column before it."""
    n, h, w, c = x.shape
    ref, scale = apply_reference(x, mean, rstd, gamma, beta, pad, relu, res)
    r = OUT_ROUND[out.dtype]
    bound = APPLY_TAU * scale * (1 + r) + r * ref.abs()
    got = out.double()
    err = (got - ref).abs()
    p = ns_plan_py(n, c, h, w, pad, h + 2 * pad, w + 2 * pad, x.element_size(), 2 if res is not None else 1, sms)
    rec = dict(nan=int(torch.isnan(got).sum()), bad=int((err > bound).sum()), ratio=_ratio(err, bound), plan=p,
               mutants={}, skipped={})

    def mut(name, m):
        rec["mutants"][name] = _ratio((got - m).abs(), bound)
    if pad:
        m = ref.clone()
        m[:, :pad], m[:, -pad:], m[:, :, :pad], m[:, :, -pad:] = 0, 0, 0, 0
        mut("zero_pad", m)
    else:
        rec["skipped"]["zero_pad"] = "pad 0"
    if res is not None:
        mut("no_res", apply_reference(x, mean, rstd, gamma, beta, pad, relu)[0])
    else:
        rec["skipped"]["no_res"] = "no residual"
    if n > 1:
        mv, rv = mean.view(n, c), rstd.view(n, c)
        k = int((mv[:-1] - mv[-1]).abs().add((rv[:-1] - rv[-1]).abs() / rv[-1]).sum(1).argmax())
        m = ref.clone()
        m[-1] = apply_reference(x[-1:], mv[k], rv[k], gamma, beta, pad, relu, None if res is None else res[-1:])[0][0]
        mut("other_image_stats", m)
    else:
        rec["skipped"]["other_image_stats"] = "one image"
    if p is not None and p["nseg"] > 1:
        m = ref.clone()
        y, oa = (h + 2 * pad) // 2, p["seg"]
        m[-1, y, oa] = ref[-1, y, oa - 1]
        mut("seam", m)
    else:
        rec["skipped"]["seam"] = "one segment"
    return rec


def check_bwd(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu, dx, gtotal, s12, sms):
    """dx, gtotal and the s12 rows of one backward call against bwd_reference.
      s1: gamma_k * sum |g'| + GPRIME_TAU * sum |terms of g'|;  s2: gamma_(k+3) * sum |g' * xhat| + GPRIME_TAU * sum
      |terms| * |xhat| (+ 2^-23 |s2| for the rstd multiply): the conditioning of the maths, k from the plan;
      gtotal = g': GPRIME_TAU * sum |terms|;  dx: DX_TAU * (|A g'| + |B| (|x| + |mean|) + |A s1| / hw) + what the s1 / s2
      bounds propagate, + the store's rounding.  Pixels whose ReLU mask depends on D's rounding add their |g|.
    Mutants: the reflect fold dropped on one border pixel of the last image, gextra dropped, the ReLU mask from x > 0,
    one row of the last image missing from the sums."""
    n, h, w, c = x.shape
    hw = h * w
    esz = x.element_size()
    nslabs = 1 + (gpad is not None) + (gextra is not None)
    p = bwd_plan(n, c, h, w, pad, esz, nslabs, sms)
    R = bwd_reference(x, mean, rstd, gamma, beta, gpad, pad, gextra, relu)
    A, xhat, gp, ga, gamb = R["A"], R["xhat"], R["gp"], R["ga"], R["gamb"]
    k = bwd_depth(p)
    b1 = gamma_k(k) * gp.abs().sum((1, 2)).flatten() + GPRIME_TAU * ga.sum((1, 2)).flatten() + gamb.sum((1, 2)).flatten()
    b2 = (gamma_k(k + 3) * (gp * xhat).abs().sum((1, 2)).flatten() + GPRIME_TAU * (ga * xhat.abs()).sum((1, 2)).flatten()
          + (gamb * xhat.abs()).sum((1, 2)).flatten() + 2 * U * R["s2"].abs())
    r = OUT_ROUND[dx.dtype]
    mu = _per_image(mean, n, c).abs()
    B = (A * _per_image(rstd, n, c) * R["s2"].view(n, 1, 1, c) / hw).abs()
    Aa = A.abs()
    bdx = (DX_TAU * (Aa * ga + B * (x.double().abs() + mu) + (Aa * R["s1"].view(n, 1, 1, c)).abs() / hw)
           + Aa * (b1.view(n, 1, 1, c) + xhat.abs() * b2.view(n, 1, 1, c)) / hw + Aa * gamb)
    bdx = bdx * (1 + r) + r * R["dx"].abs()
    bgt = (GPRIME_TAU * ga + gamb) * (1 + r) + r * gp.abs()
    gdx = dx.double()
    gs1, gs2 = s12[0].double(), s12[1].double()
    outs = [(gdx, R["dx"], bdx), (gs1, R["s1"], b1), (gs2, R["s2"], b2)]
    ggt = None
    if gtotal is not None:
        ggt = gtotal.double()
        outs.append((ggt, gp, bgt))
    rec = dict(plan=p, k=k, amb=R["amb"], mutants={}, skipped={},
               nan=int(torch.isnan(gdx).sum()) + (0 if ggt is None else int(torch.isnan(ggt).sum())),
               bad=sum(int(((g - want).abs() > b).sum()) for g, want, b in outs),
               ratio=max(_ratio((g - want).abs(), b) for g, want, b in outs),
               ratio_dx=_ratio((gdx - R["dx"]).abs(), bdx),
               ratio_sums=max(_ratio((gs1 - R["s1"]).abs(), b1), _ratio((gs2 - R["s2"]).abs(), b2)))

    def mut(name, gp_m, s1_m=None, s2_m=None):
        if s1_m is None:
            s1_m, s2_m = bwd_sums(gp_m, xhat)
        want = [bwd_dx(gp_m, xhat, A, s1_m, s2_m, n, c, hw), s1_m, s2_m] + ([gp_m] if ggt is not None else [])
        rec["mutants"][name] = max(_ratio((g - m).abs(), b) for (g, _, b), m in zip(outs, want))

    mask = R["mask"]
    if pad and gpad is not None:
        centre = gpad[:, pad:pad + h, pad:pad + w].double()
        extra = gextra.double() if gextra is not None else 0.0
        delta = (R["g"] - centre - extra) * mask                             # what the fold adds
        score = (Aa * delta.abs() / bdx.clamp_min(1e-300))[-1].amax(-1)       # [h, w] of the last image
        i, j = divmod(int(score.flatten().argmax()), w)
        gp_m = gp.clone()
        gp_m[-1, i, j] -= delta[-1, i, j]
        mut("fold_pixel", gp_m, R["s1"], R["s2"])                              # one pixel: the sums barely move
        rec["fold_pixel"] = (i, j)
    else:
        rec["skipped"]["fold_pixel"] = "no padded gradient" if gpad is None else "pad 0"
    if gextra is not None:
        mut("no_gextra", gp - gextra.double() * mask)
    else:
        rec["skipped"]["no_gextra"] = "no gextra"
    if relu:
        mut("mask_from_x", R["g"] * (x.double() > 0))
    else:
        rec["skipped"]["mask_from_x"] = "no ReLU"
    rows1 = gp[-1].sum(1)                                                    # [h, c]: per row of the last image
    rows2 = (gp[-1] * xhat[-1]).sum(1)
    b1l, b2l = b1.view(n, c)[-1], b2.view(n, c)[-1]
    i = int(torch.maximum(rows1.abs() / b1l.clamp_min(1e-300), rows2.abs() / b2l.clamp_min(1e-300)).amax(1).argmax())
    s1_m, s2_m = R["s1"].clone().view(n, c), R["s2"].clone().view(n, c)
    s1_m[-1] -= rows1[i]
    s2_m[-1] -= rows2[i]
    mut("row_missing", gp, s1_m.flatten(), s2_m.flatten())
    rec["row_missing"] = i
    return rec


# ---------------------------------------------------------------------------------------------------------------------
# The probe.

class _NormProbe:
    """Wraps ops.instnorm_finalize / instnorm_stats / instnorm_apply / instnorm_bwd: NaN in the outputs, a snapshot of
    the storage around them, clones of the inputs and the family counters; then the real call, once, with unchanged
    arguments, a synchronise and the fp64 checks.  Asserts come after the run."""

    NAMES = ("instnorm_finalize", "instnorm_stats", "instnorm_apply", "instnorm_bwd")

    def __init__(self, lib, ops, sms):
        self.lib, self.sms = lib, sms
        self.real = {name: getattr(ops, name) for name in self.NAMES}
        self.recs = []

    def _bind(self, name, args, kwargs):
        a = inspect.signature(self.real[name]).bind(*args, **kwargs)
        a.apply_defaults()
        return a.arguments

    def _run(self, name, args, kwargs, inputs):
        clones = {k: t.clone() for k, t in inputs.items() if t is not None}
        fam0 = self.lib.family_stats()
        res = self.real[name](*args, **kwargs)
        torch.cuda.synchronize()
        fam = self.lib.family_delta(fam0)
        changed = [k for k, t in clones.items() if not torch.equal(_bits(inputs[k]), _bits(t))]
        fams = {f: v[0] for f, v in fam.items() if v[0]}
        return res, dict(site=_site(), inputs_changed=changed, fams=fams)

    def instnorm_finalize(self, *args, **kwargs):
        a = self._bind("instnorm_finalize", args, kwargs)
        sums = a["sums"]
        (mean, rstd), rec = self._run("instnorm_finalize", args, kwargs, dict(sums=sums))
        rec.update(entry="finalize", want=dict(in_stats=1), n=a["n"], c=a["c"], hw=a["hw"], sums=sums.clone(),
                   mean=mean, rstd=rstd, eps=a["eps"], shape=(a["n"], a["c"], a["hw"]))
        self.recs.append(rec)        # checked once the apply call that reads this mean tells the image width
        return mean, rstd

    def instnorm_stats(self, *args, **kwargs):
        a = self._bind("instnorm_stats", args, kwargs)
        x = a["x"]
        (mean, rstd), rec = self._run("instnorm_stats", args, kwargs, dict(x=x))
        rec.update(entry="stats", want=dict(in_stats=1), shape=(tuple(x.shape), str(x.dtype)[6:]),
                   **check_stats(x, mean, rstd, self.sms, a["eps"]))
        self.recs.append(rec)
        return mean, rstd

    def instnorm_apply(self, *args, **kwargs):
        a = self._bind("instnorm_apply", args, kwargs)
        x, out, res = a["x"], a["out"], a["residual"]
        out.fill_(float("nan"))
        st = _storage_view(out)
        before = st.clone()
        ins = dict(x=x, mean=a["mean"], rstd=a["rstd"], gamma=a["gamma"], beta=a["beta"], res=res)
        result, rec = self._run("instnorm_apply", args, kwargs, ins)
        rec.update(entry="apply", want=dict(in_apply=1), shape=(tuple(x.shape), str(x.dtype)[6:], a["pad"],
                   bool(a["relu"]), res is not None), mean_ptr=a["mean"].data_ptr(), hw=(x.shape[1], x.shape[2]),
                   changed_outside=_changed_outside(before, st, _inside(out, lambda v: v.fill_(True))),
                   **check_apply(x, a["mean"], a["rstd"], a["gamma"], a["beta"], res, out, a["pad"], a["relu"],
                                 self.sms))
        for f in self.recs[::-1]:                      # the finalize call whose mean this is
            if f["entry"] == "finalize" and "bad" not in f and f["mean"].data_ptr() == rec["mean_ptr"]:
                rec_f = check_finalize(f["sums"], f["n"], f["c"], f["hw"], f["mean"], f["rstd"], f["eps"],
                                       row=x.shape[2])
                f.update(rec_f, hw_match=f["hw"] == x.shape[1] * x.shape[2], skipped={})
                del f["sums"]
                break
        self.recs.append(rec)
        return result

    def instnorm_bwd(self, *args, **kwargs):
        a = self._bind("instnorm_bwd", args, kwargs)
        x, dx, gtotal, s12, arrive = a["x"], a["dx"], a["gtotal"], a["s12"], a["arrive"]
        assert s12 is not None and arrive is not None, "the step passes its shared sums buffer"
        zero_on_entry = bool((s12 == 0).all()) and bool((arrive == 0).all())
        outs = [t for t in (dx, gtotal) if t is not None]
        for t in outs:
            t.fill_(float("nan"))
        snaps = [(t, _storage_view(t), _storage_view(t).clone()) for t in outs]
        bank = _storage_view(s12)
        bank_before = bank.clone()
        ins = dict(x=x, mean=a["mean"], rstd=a["rstd"], gamma=a["gamma"], beta=a["beta"], gpad=a["gpad"],
                   gextra=a["gextra"])
        result, rec = self._run("instnorm_bwd", args, kwargs, ins)
        changed = sum(_changed_outside(b, s, _inside(t, lambda v: v.fill_(True))) for t, s, b in snaps)
        inside = _inside(s12, lambda v: v.fill_(True))
        if arrive.untyped_storage().data_ptr() == s12.untyped_storage().data_ptr():
            inside |= _inside(arrive, lambda v: v.fill_(True))
        rec.update(entry="bwd", shape=(tuple(x.shape), str(x.dtype)[6:], a["pad"], bool(a["relu"]),
                   a["gpad"] is not None, a["gextra"] is not None, gtotal is not None),
                   changed_outside=changed + _changed_outside(bank_before, bank, inside), zero_on_entry=zero_on_entry,
                   arrive=(int(arrive.min()), int(arrive.max())),
                   **check_bwd(x, a["mean"], a["rstd"], a["gamma"], a["beta"], a["gpad"], a["pad"], a["gextra"],
                               a["relu"], dx, gtotal, s12, self.sms))
        rec["want"] = dict(in_bwd=rec["plan"]["launches"])
        self.recs.append(rec)
        return result


def probe_failures(rec):
    """Everything wrong with one call's record (empty when it passed)."""
    f = []
    if rec["entry"] == "finalize" and "bad" not in rec:
        return ["no apply call read this mean, so it was never checked"]
    if rec["fams"] != rec["want"]:
        f.append(f"launches {rec['fams']}, expected {rec['want']}")
    if rec["inputs_changed"]:
        f.append(f"inputs changed: {rec['inputs_changed']}")
    if rec["bad"]:
        f.append(f"{rec['bad']} values over the bound (max err/bound {rec['ratio']:.2e})")
    if rec.get("nan"):
        f.append(f"{rec['nan']} output elements not written")
    if rec.get("changed_outside"):
        f.append(f"{rec['changed_outside']} elements outside the outputs changed")
    if rec["entry"] == "finalize" and not rec["hw_match"]:
        f.append(f"hw {rec['hw']} is not the plane the apply normalises")
    if rec["entry"] == "bwd":
        if not rec["zero_on_entry"]:
            f.append("s12 / arrive not zero on entry")
        want = (rec["plan"]["nblk"],) * 2 if rec["plan"]["launches"] == 1 else (0, 0)
        if rec["arrive"] != want:
            f.append(f"barrier counters {rec['arrive']}, the plan says {want}")
    for k, v in rec["mutants"].items():
        if not v > 1:
            f.append(f"mutant {k} stays within the bound ({v:.2f}x)")
    return f


def _fmt(rec):
    mut = ", ".join(f"{k} {v:.1f}x" for k, v in sorted(rec["mutants"].items())) or "-"
    skip = "; ".join(f"{k} n/a ({v})" for k, v in sorted(rec.get("skipped", {}).items()))
    plan = rec.get("plan")
    pl = ""
    if plan and "nseg" in plan:
        pl = f" plan nblk={plan['nblk']} nseg={plan['nseg']} seg={plan['seg']}" + (
            f" launches={plan['launches']} k={rec['k']}" if "launches" in plan else "")
    return (f"{rec['entry']} {rec['site']} {rec.get('shape')}{pl}: max err/bound {rec.get('ratio', float('nan')):.2e}; "
            f"mutants {mut}" + (f"; {skip}" if skip else ""))


@pytest.fixture(scope="module")
def ast():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import artist_style_transfer_b200 as m
    return m


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _report(tag, probe, step, t0):
    fails = []
    worst = {}
    for i, rec in enumerate(probe.recs):
        print(f"[{tag}] #{i} {_fmt(rec)}")
        worst[rec["entry"]] = max(worst.get(rec["entry"], 0.0), rec.get("ratio", float("nan")))
        fails += [f"#{i} {rec['entry']} {rec['site']}: {e}" for e in probe_failures(rec)]
    seen = {}
    for rec in probe.recs:
        for f, v in rec["fams"].items():
            seen[f] = seen.get(f, 0) + v
    ran = {f: step[f][0] for f in IN_FAMILIES if step[f][0]}
    if {f: v for f, v in seen.items() if f in IN_FAMILIES} != ran:
        fails.append(f"the run launched {ran}, the probes saw {seen}")
    print(f"[{tag}] worst err/bound per call type {({k: f'{v:.2e}' for k, v in worst.items()})}; InstanceNorm launches "
          f"{ran}; wall time {time.time() - t0:.1f} s")
    return fails, ran


@pytest.mark.gpu
@pytest.mark.parametrize("mode,batch,h,w", WORKLOADS, ids=[f"{m}-b{b}-{h}x{w}" for m, b, h, w in WORKLOADS])
def test_instnorm_launches_of_a_step(ast, monkeypatch, mode, batch, h, w):
    from artist_style_transfer_b200 import _lib, ops
    from oracle import weights
    t0 = time.time()
    net, vgg = _build(ast, mode)
    content = weights.content_batch(batch, h, 2, width=w).cuda()
    style = ast.style_grams_single(vgg, weights.style_image(h, 2).cuda(), batch)
    probe = _NormProbe(_lib, ops, _sms())
    for name in probe.NAMES:
        monkeypatch.setattr(ops, name, getattr(probe, name))
    fam0 = _lib.family_stats()
    ast.perceptual_step(net, vgg, content, style)        # eager: the probes synchronise, which graph capture forbids
    torch.cuda.synchronize()
    step = _lib.family_delta(fam0)
    monkeypatch.undo()
    fails, ran = _report(f"{mode} B={batch} {h}x{w}", probe, step, t0)
    by = {e: [r for r in probe.recs if r["entry"] == e] for e in ("finalize", "stats", "apply", "bwd")}
    n_norm = len(by["apply"])
    if len(by["bwd"]) != n_norm or len(by["finalize"]) + len(by["stats"]) != n_norm:
        fails.append(f"{n_norm} apply calls, {len(by['bwd'])} backward calls, {len(by['finalize'])} finalize and "
                     f"{len(by['stats'])} stats calls")
    if mode == "fp32" and by["finalize"]:
        fails.append(f"strict mode finalized {len(by['finalize'])} fused statistics")
    if (mode, batch, h, w) == ("fast", 32, 256, 256):
        single = sum(r["plan"]["launches"] == 1 for r in by["bwd"])
        got = dict(in_apply=ran.get("in_apply", 0), bwd_single=single, bwd_double=len(by["bwd"]) - single)
        if got != STEP_B32 or ran.get("in_bwd") != STEP_B32["bwd_single"] + 2 * STEP_B32["bwd_double"]:
            fails.append(f"InstanceNorm launches {got} ({ran}), DESIGN section 5 states {STEP_B32}")
    assert probe.recs and not fails, "\n".join(fails)


@pytest.mark.gpu
def test_instnorm_launches_of_stylize_1080p(ast, monkeypatch):
    """The forward of a 1080x1920 frame: its last apply writes 1928 padded columns (C=32, pad 4) in eight segments."""
    from artist_style_transfer_b200 import _lib, ops
    from oracle import weights
    t0 = time.time()
    net = ast.StyleTransfer(device=torch.device("cuda"), precision="fast")
    net.load_state_dict(weights.transfer_state_dict(2), strict=True)
    g = torch.Generator().manual_seed(5)
    frame = torch.randint(0, 256, (1, 1080, 1920, 3), dtype=torch.uint8, generator=g).cuda()
    probe = _NormProbe(_lib, ops, _sms())
    for name in probe.NAMES:
        monkeypatch.setattr(ops, name, getattr(probe, name))
    fam0 = _lib.family_stats()
    net.stylize(frame)
    torch.cuda.synchronize()
    step = _lib.family_delta(fam0)
    monkeypatch.undo()
    fails, _ = _report("stylize fast 1080x1920", probe, step, t0)
    wide = [r for r in probe.recs if r["entry"] == "apply" and r["plan"]["width"] == 1928]
    if not wide or wide[-1]["plan"]["nseg"] != 8 or "seam" not in wide[-1]["mutants"]:
        fails.append(f"no apply call over 1928 columns in 8 segments: {[r['plan'] for r in wide]}")
    if any(r["entry"] == "bwd" for r in probe.recs):
        fails.append("stylize ran a backward")
    assert probe.recs and not fails, "\n".join(fails)


# ---------------------------------------------------------------------------------------------------------------------
# Standalone calls at the edges of the staging plan.

APPLY_CASES = [
    # (dtype, n, h, w, c, pad, relu, residual)
    ("bf16", 2, 9, 252, 32, 1, True, False),     # 254 padded columns = seg_max: one segment
    ("bf16", 2, 9, 253, 32, 1, True, True),      # 255: two segments, the reflect border on the seam's far side
    ("bf16", 2, 16, 70, 128, 1, False, True),    # two segments of 36 columns
    ("bf16", 2, 5, 5, 32, 4, True, True),        # pad 4, h = w = pad + 1: every pixel is mirrored
    ("fp32", 2, 5, 5, 4, 4, False, False),
    ("bf16", 2, 64, 64, 8, 1, True, False),      # 1 lane, 256 slots
    ("bf16", 2, 16, 16, 1024, 1, True, True),    # 128 lanes, 2 slots, 6-column segments
    ("fp32", 3, 32, 32, 4, 1, True, True),
    ("fp32", 2, 16, 16, 512, 1, False, False),
    ("bf16", 1, 300, 40, 32, 1, True, False),    # n = 1: one row per block
    ("bf16", 300, 8, 8, 32, 1, True, True),      # n = 300: one block per image
    ("fp32", 2, 24, 2000, 32, 4, True, False),   # 2008 padded fp32 columns: 17 segments
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt,n,h,w,c,pad,relu,res", APPLY_CASES)
def test_instnorm_apply_plan_edges(ast, dt, n, h, w, c, pad, relu, res):
    from artist_style_transfer_b200 import _lib, ops
    torch.manual_seed(n * 7 + h + c)
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    x = (torch.randn(n, h, w, c, device="cuda") * 2 + 0.5).to(dtype)
    m, r, _ = stats_reference(x)
    mean, rstd = m.float(), r.float()
    gamma = torch.rand(c, device="cuda") + 0.5
    beta = torch.randn(c, device="cuda") * 0.3
    rt = torch.randn(n, h, w, c, device="cuda").to(dtype) if res else None
    buf = torch.full((n * (h + 2 * pad) * (w + 2 * pad) * c + 64,), 7.0, dtype=dtype, device="cuda")
    out = buf[32:32 + n * (h + 2 * pad) * (w + 2 * pad) * c].view(n, h + 2 * pad, w + 2 * pad, c)
    out.fill_(float("nan"))
    before = buf.clone()
    fam0 = _lib.family_stats()
    ops.instnorm_apply(x, mean, rstd, gamma, beta, out, pad, relu, residual=rt)
    torch.cuda.synchronize()
    launches = {f: v[0] for f, v in _lib.family_delta(fam0).items() if v[0]}
    rec = check_apply(x, mean, rstd, gamma, beta, rt, out, pad, relu, _sms())
    rec.update(site="standalone", entry="apply", shape=(n, h, w, c, dt, pad))
    print(_fmt(rec))
    assert launches == {"in_apply": 1}
    assert rec["nan"] == 0 and rec["bad"] == 0, rec
    assert _changed_outside(before, buf, _inside(out, lambda v: v.fill_(True))) == 0
    assert all(v > 1 for v in rec["mutants"].values()), rec["mutants"]
    assert ("seam" in rec["mutants"]) == (rec["plan"]["nseg"] > 1)


STATS_CASES = [
    # (dtype, n, h, w, c, mean, std)
    ("fp32", 2, 64, 64, 128, 300.0, 1.0),        # |mean| / std = 300: the E[x^2] - mean^2 cancellation case
    ("bf16", 2, 64, 64, 64, 100.0, 0.5),
    ("fp32", 3, 5, 7, 128, 0.5, 2.0),            # hw = 35 < 64 slots: most threads see no pixel
    ("fp32", 2, 33, 31, 24, 1.0, 1.0),           # C = 24: 6 lanes, 42 slots, 4 idle threads
    ("fp32", 1, 1024, 1024, 32, -2.0, 3.0),
    ("bf16", 300, 8, 8, 32, 1.0, 1.0),
    ("fp32", 2, 16, 16, 1024, 0.0, 1.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt,n,h,w,c,mu,sd", STATS_CASES)
def test_instnorm_strict_statistics(ast, dt, n, h, w, c, mu, sd):
    from artist_style_transfer_b200 import _lib, ops
    torch.manual_seed(n + h + c)
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    x = (torch.randn(n, h, w, c, device="cuda") * sd + mu).to(dtype)
    xc = x.clone()
    fam0 = _lib.family_stats()
    mean, rstd = ops.instnorm_stats(x)
    torch.cuda.synchronize()
    assert {f: v[0] for f, v in _lib.family_delta(fam0).items() if v[0]} == {"in_stats": 1}
    rec = check_stats(x, mean, rstd, _sms())
    print(f"stats {dt} {(n, h, w, c)} |mean|/std {rec['mu_sd']:.0f}: max err/bound {rec['ratio']:.2e}, "
          f"max |d rstd|/rstd {rec['rel_rstd']:.1e}, plan {rec['plan']}")
    assert torch.equal(_bits(x), _bits(xc))
    assert rec["bad"] == 0, rec


def test_staged_kernels_refuse_what_they_cannot_split():
    """C = 24 fp32: the statistics take it (6 lanes of 4 channels), apply refuses it (256 consumers do not split into 6
    lanes) before any CUDA call."""
    import ctypes
    from artist_style_transfer_b200 import _lib
    lib = _lib.load()
    n, h, w, c, pad = 2, 8, 8, 24, 1
    x = _lib.Image(1 << 20, _lib.AST_F32, n, h, w, c, h * w * c, w * c, c, 1)
    out = _lib.Image(1 << 20, _lib.AST_F32, n, h + 2, w + 2, c, (h + 2) * (w + 2) * c, (w + 2) * c, c, 1)
    p = ctypes.c_void_p(1 << 20)
    rc = lib.ast_instnorm_apply(ctypes.byref(x), p, p, p, p, None, ctypes.byref(out), pad, 1, None)
    assert rc < 0 and b"C=24 is not supported" in lib.ast_last_error(), lib.ast_last_error()
