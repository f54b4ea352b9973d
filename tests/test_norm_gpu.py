"""BatchNorm / activation kernels of csrc/norm.cu called directly, each against a plain float64 reference on the
same bf16-rounded inputs (torch on the GPU in float64; autograd through F.batch_norm for the backward).

Gates are per element, not over whole vectors:
  * bf16 outputs: within one bf16 ulp of the reference, plus 1e-4 x the sum of the absolute values of the terms
    where the output is a sum that cancels (normalise: x*scale + shift; backward: scale*g + k1*z + k0);
  * fp32 reductions (statistics, dgamma, dbeta, dbias): |err| <= 1e-5 * sum |terms| + 1e-6;
  * ReLU / LeakyReLU masks come from the coefficients the kernel itself used: a sign flip at 0 is not an error.
Every kernel that writes a view also runs with its output as a channel slice of a sentinel-filled buffer, and
every accumulating output is checked to accumulate."""
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import assert_bf16, assert_f32_sum, assert_within

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64
DEV = "cuda"
SENTINEL = -7.0
EPS = 1e-5
MOMENTUM = 0.1


# ------------------------------------------------------------------ views
def nhwc(npix, c, ld=None, off=0, fill=SENTINEL):
    """(buffer [1, 1, npix, ld], its channel slice [off, off + c)) -- the kernels' (pointer, ld) views."""
    ld = ld or c
    buf = torch.full((1, 1, npix, ld), fill, device=DEV, dtype=BF)
    return buf, buf[..., off:off + c]


def rand_view(g, npix, c, ld=None, off=0, scale=1.0, offset=None):
    buf, v = nhwc(npix, c, ld, off)
    x = torch.randn(1, 1, npix, c, device=DEV, generator=g) * scale
    if offset is not None:
        x = x + offset
    v.copy_(x.to(BF))
    return buf, v


def assert_outside_untouched(name, buf, off, c):
    outside = torch.ones(buf.shape[-1], dtype=torch.bool, device=DEV)
    outside[off:off + c] = False
    assert bool((buf[..., outside].float() == SENTINEL).all()), name + ": wrote outside its channel slice"


def block_for(c):
    """Threads per block of the streaming BatchNorm kernels (csrc/norm.cu block_for)."""
    groups = c // 8
    return (256 // groups) * groups or groups


def act_mask_grad(pre64, act, slope):
    """act'(pre) where pre is the exact value of the kernel's fp32 z*scale + shift."""
    if act == 0:
        return torch.ones_like(pre64)
    neg = 0.0 if act == 1 else slope
    return torch.where(pre64 > 0, torch.ones_like(pre64), torch.full_like(pre64, neg))


def act_apply(y, mask_pre, act, slope):
    if act == 0:
        return y
    return torch.where(mask_pre > 0, y, y * (0.0 if act == 1 else slope))


def flat(v):
    return v.reshape(-1, v.shape[-1])


# ------------------------------------------------------------------ channel_stats
STATS_C = [8, 24, 64, 96, 512, 2048]
STATS_NPIX = ["1", "py-1", "4py+3", "large"]


def stats_npix(c, kind):
    py = block_for(c) // (c // 8)
    return {"1": 1, "py-1": max(py - 1, 1), "4py+3": 4 * py + 3, "large": (1 << 23) // c + 5}[kind]


@pytest.mark.parametrize("c", STATS_C)
@pytest.mark.parametrize("kind", STATS_NPIX)
def test_channel_stats(cuda_lib, c, kind):
    from dasemanticsegmentationaml_b200 import kernels as K
    npix = stats_npix(c, kind)
    g = torch.Generator(device=DEV).manual_seed(c * 7 + npix)
    ld, off = (c + 16, 8) if kind != "large" else (c, 0)
    offset = torch.randn(c, device=DEV, generator=g)
    _, x = rand_view(g, npix, c, ld, off, offset=offset)
    stats = torch.zeros(2, c, device=DEV)
    K.channel_stats(x, stats)
    x64 = flat(x).double()
    want = torch.stack([x64.sum(0), (x64 * x64).sum(0)])
    terms = torch.stack([x64.abs().sum(0), (x64 * x64).sum(0)])
    assert_f32_sum("channel_stats C%d npix%d" % (c, npix), stats, want, terms)
    K.channel_stats(x, stats)   # accumulates
    assert_f32_sum("channel_stats C%d npix%d twice" % (c, npix), stats, 2 * want, 2 * terms)


# ------------------------------------------------------------------ forward: bn_norm_act / bn_finalize + bn_act_apply
FWD_CASES = [
    # c, npix, act, affine, view
    (8, 1029, 1, True, False),
    (24, 4099, 2, True, True),
    (40, 777, 0, False, True),
    (96, 2311, 1, False, False),
    (512, 1031, 2, True, True),
    (2048, 130, 1, True, False),
    (64, 1, 2, True, False),
]


def bn_reference(x64, count, gamma, beta, rm0, rv0):
    """float64 F.batch_norm(training=True) on [npix, C]: output, batch mean / biased var, running stats."""
    rm, rv = rm0.double().clone(), rv0.double().clone()
    g64 = None if gamma is None else gamma.double()
    b64 = None if beta is None else beta.double()
    mean = x64.mean(0)
    var = x64.var(0, unbiased=False)
    if count > 1:
        y = F.batch_norm(x64, rm, rv, g64, b64, training=True, momentum=MOMENTUM, eps=EPS)
    else:   # torch refuses one value per channel in training mode; the unbiased variance is taken as 0 then
        y = (x64 - mean) / torch.sqrt(var + EPS) * (1.0 if g64 is None else g64) + (0.0 if b64 is None else b64)
        rm.mul_(1 - MOMENTUM).add_(MOMENTUM * mean)
        rv.mul_(1 - MOMENTUM)
    return y, mean, var, rm, rv


@pytest.mark.parametrize("case", FWD_CASES, ids=lambda c: "C%d-px%d-act%d-%s%s" % (
    c[0], c[1], c[2], "affine" if c[3] else "nogamma", "-view" if c[4] else ""))
def test_bn_norm_act_train(cuda_lib, case):
    from dasemanticsegmentationaml_b200 import kernels as K
    c, npix, act, affine, view = case
    slope = 0.2
    g = torch.Generator(device=DEV).manual_seed(c + npix)
    ld, off = (c + 24, 16) if view else (c, 0)
    _, x = rand_view(g, npix, c, ld, off, offset=0.5 * torch.randn(c, device=DEV, generator=g))
    gamma = torch.rand(c, device=DEV, generator=g) + 0.5 if affine else None
    beta = torch.randn(c, device=DEV, generator=g) if affine else None
    rm0 = torch.randn(c, device=DEV, generator=g)
    rv0 = torch.rand(c, device=DEV, generator=g) + 0.5
    x64 = flat(x).double()
    stats = torch.stack([x64.sum(0), (x64 * x64).sum(0)]).float()   # exact sums, rounded once
    ybuf, y = nhwc(npix, c, ld, off)
    rm, rv = rm0.clone(), rv0.clone()
    scale, shift, mean, rstd = (torch.full((c,), float("nan"), device=DEV) for _ in range(4))
    K.bn_norm_act(x, y, stats, float(npix), gamma, beta, rm, rv, True, act, slope, scale, shift, mean, rstd,
                  momentum=MOMENTUM, eps=EPS)
    yr, mr, vr, rmr, rvr = bn_reference(x64, npix, gamma, beta, rm0, rv0)
    name = "bn_norm_act C%d px%d act%d" % (c, npix, act)
    ex2 = (x64 * x64).mean(0)
    # var = E[x^2] - mean^2 in fp32: its error is relative to E[x^2] + mean^2, not to var
    var_terms = ex2 + mr * mr
    assert_within(name + " mean", mean, mr, 1e-5 * x64.abs().mean(0) + 1e-6)
    rstd_r = 1.0 / torch.sqrt(vr + EPS)
    assert_within(name + " rstd", rstd, rstd_r, rstd_r * (1e-5 * var_terms / (vr + EPS) + 1e-6))
    g64 = gamma.double() if affine else torch.ones_like(mr)
    b64 = beta.double() if affine else torch.zeros_like(mr)
    assert_within(name + " scale", scale, g64 * rstd_r, (g64 * rstd_r).abs() * (1e-5 * var_terms / (vr + EPS) + 1e-6))
    assert_within(name + " shift", shift, b64 - mr * g64 * rstd_r,
                  1e-5 * (b64.abs() + (mr * g64 * rstd_r).abs() * (1 + var_terms / (vr + EPS))) + 1e-6)
    # running statistics: momentum 0.1 and the UNBIASED batch variance (count / (count - 1))
    assert_within(name + " running_mean", rm, rmr, 1e-5 * (0.9 * rm0.double().abs() + 0.1 * x64.abs().mean(0)) + 1e-6)
    bessel = npix / (npix - 1.0) if npix > 1 else 1.0
    assert_within(name + " running_var", rv, rvr, 1e-5 * (0.9 * rv0.double() + 0.1 * var_terms * bessel) + 1e-6)
    # output: the activation mask from the kernel's own published scale / shift
    pre_k = x64 * scale.double() + shift.double()
    want = act_apply(yr, pre_k, act, slope)
    terms = (x64 * scale.double()).abs() + shift.double().abs()
    assert_bf16(name + " y", flat(y), want, terms)
    if view:
        assert_outside_untouched(name, ybuf, off, c)

    # the two-launch path: bn_finalize + bn_act_apply agree with the fused launch
    rm2, rv2 = rm0.clone(), rv0.clone()
    sc2, sh2, m2, r2 = (torch.full((c,), float("nan"), device=DEV) for _ in range(4))
    K.bn_finalize(stats, float(npix), gamma, beta, rm2, rv2, True, sc2, sh2, m2, r2, momentum=MOMENTUM, eps=EPS)
    y2buf, y2 = nhwc(npix, c, ld, off)
    K.bn_act_apply(x, y2, sc2, sh2, act, slope)
    for nm, a, b in (("scale", sc2, scale), ("shift", sh2, shift), ("mean", m2, mean), ("rstd", r2, rstd),
                     ("running_mean", rm2, rm), ("running_var", rv2, rv)):
        assert_within(name + " finalize " + nm, a, b, b.double().abs() * 2.0 ** -22 + 1e-30)
    pre2 = x64 * sc2.double() + sh2.double()
    assert_bf16(name + " apply y", flat(y2), act_apply(yr, pre2, act, slope), terms)
    if view:
        assert_outside_untouched(name + " apply", y2buf, off, c)


@pytest.mark.parametrize("c,act", [(24, 1), (256, 2), (64, 0)])
def test_bn_norm_act_eval(cuda_lib, c, act):
    """Eval mode: coefficients from the running statistics, which stay untouched."""
    from dasemanticsegmentationaml_b200 import kernels as K
    npix, slope = 3001, 0.2
    g = torch.Generator(device=DEV).manual_seed(c)
    _, x = rand_view(g, npix, c, c + 8, 8)
    gamma = torch.rand(c, device=DEV, generator=g) + 0.5
    beta = torch.randn(c, device=DEV, generator=g)
    rm0 = torch.randn(c, device=DEV, generator=g)
    rv0 = torch.rand(c, device=DEV, generator=g) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    ybuf, y = nhwc(npix, c, c + 8, 0)
    scale, shift, mean, rstd = (torch.full((c,), float("nan"), device=DEV) for _ in range(4))
    K.bn_norm_act(x, y, None, float(npix), gamma, beta, rm, rv, False, act, slope, scale, shift, mean, rstd)
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
    x64 = flat(x).double()
    yr = F.batch_norm(x64, rm0.double(), rv0.double(), gamma.double(), beta.double(), training=False, eps=EPS)
    rstd_r = 1.0 / torch.sqrt(rv0.double() + EPS)
    assert_within("eval mean", mean, rm0.double(), torch.full_like(rstd_r, 1e-30))
    assert_within("eval rstd", rstd, rstd_r, rstd_r * 1e-6)
    pre_k = x64 * scale.double() + shift.double()
    terms = (x64 * scale.double()).abs() + shift.double().abs()
    assert_bf16("eval y C%d" % c, flat(y), act_apply(yr, pre_k, act, slope), terms)
    assert_outside_untouched("eval y", ybuf, 0, c)
    # bn_finalize in eval mode: the same coefficients, running statistics untouched
    sc2, sh2 = torch.empty(c, device=DEV), torch.empty(c, device=DEV)
    K.bn_finalize(None, float(npix), gamma, beta, rm, rv, False, sc2, sh2, None, None)
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
    assert_within("eval finalize scale", sc2, scale, scale.double().abs() * 2.0 ** -22)
    assert_within("eval finalize shift", sh2, shift, shift.double().abs() * 2.0 ** -22 + 1e-30)


# ------------------------------------------------------------------ backward
def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def fused_thresholds(c):
    """Pixel counts at which b200_bn_act_bwd_fused (csrc/norm.cu) switches template instance: it runs U pixels per
    batch with U = 4 (no dy2) when blocks_at(4) >= cap0, else U = 2 when blocks_at(2) >= cap0, else 1, where
    blocks_at(u) = ceil(npix / (py * u)), py = block_for(C) / (C / 8) and cap0 = 2 CTAs x SM count.  So
    blocks_at(u) >= cap0  <=>  npix >= (cap0 - 1) * py * u + 1."""
    py = block_for(c) // (c // 8)
    cap0 = 2 * n_sm()
    return {2: (cap0 - 1) * py * 2 + 1, 4: (cap0 - 1) * py * 4 + 1}


def fused_instance(c, npix, dy2):
    """(U, fold) the launcher picks: the same rule as fused_thresholds, and the warp-shuffle fold of the block
    reduction that runs when the channel-group count divides 32 and blocks are whole warps."""
    t = fused_thresholds(c)
    if not dy2 and npix >= t[4]:
        u = 4
    elif npix >= t[2]:
        u = 2
    else:
        u = 1
    groups = c // 8
    return u, groups < 32 and 32 % groups == 0 and block_for(c) % 32 == 0


BWD_C = [24, 32, 40, 96, 128, 256, 1024, 2048]
# (dy2 given, expected U, where npix sits relative to the thresholds)
BWD_POINTS = [(False, 1, "n2-1"), (False, 2, "n2"), (False, 2, "n4-1"), (False, 4, "n4"),
              (True, 1, "n2-1"), (True, 2, "n2")]
FOLD_C = (8, 16, 32, 64, 128)


def _bwd_id(c, point):
    dy2, u, where = point
    return "C%d-%s-u%d-%s-at_%s" % (c, "dy2" if dy2 else "nody2", u, "fold" if c in FOLD_C else "nofold", where)


BWD_CASES = [pytest.param(c, p, id=_bwd_id(c, p)) for c in BWD_C for p in BWD_POINTS]


def bwd_inputs(g, c, npix, dy2, view):
    """z (a BatchNorm input), its float64 batch statistics rounded to the fp32 coefficients the forward publishes,
    and the incoming gradients; views place every tensor in a channel slice of a wider buffer."""
    lds = (c + 8, c + 16, c + 24, c + 32) if view else (c, c, c, c)
    offs = (8, 0, 16, 24) if view else (0, 0, 0, 0)
    _, z = rand_view(g, npix, c, lds[0], offs[0], offset=0.5 * torch.randn(c, device=DEV, generator=g))
    _, d1 = rand_view(g, npix, c, lds[1], offs[1])
    d2 = rand_view(g, npix, c, lds[2], offs[2])[1] if dy2 else None
    dzbuf, dz = nhwc(npix, c, lds[3], offs[3])
    z64 = flat(z).double()
    mean64 = z64.mean(0)
    rstd64 = 1.0 / torch.sqrt(z64.var(0, unbiased=False) + EPS)
    gamma = torch.rand(c, device=DEV, generator=g, dtype=F64) + 0.5
    beta = torch.randn(c, device=DEV, generator=g, dtype=F64)
    coeff = dict(scale=(gamma * rstd64).float(), shift=(beta - mean64 * gamma * rstd64).float(),
                 mean=mean64.float(), rstd=rstd64.float())
    return z, d1, d2, dz, dzbuf, offs[3], gamma, beta, coeff


def bwd_reference(z, d1, d2, gamma, beta, coeff, act, slope):
    """float64 autograd through F.batch_norm(training=True); act' from the kernel's fp32 z*scale + shift."""
    z64 = flat(z).double().requires_grad_(True)
    gm, bt = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    y = F.batch_norm(z64, None, None, gm, bt, training=True, eps=EPS)
    dy = flat(d1).double() + (flat(d2).double() if d2 is not None else 0.0)
    pre_k = z64.detach() * coeff["scale"].double() + coeff["shift"].double()
    gg = dy * act_mask_grad(pre_k, act, slope)
    y.backward(gg)
    return z64.grad, gm.grad, bt.grad, gg, pre_k


def check_bwd(name, z, dz, red0, coeff, ref, gg, pre_k, npix):
    dz_r, dgamma_r, dbeta_r = ref
    z64 = flat(z).double()
    sc, mu, rs = coeff["scale"].double(), coeff["mean"].double(), coeff["rstd"].double()
    # dz = sc*g + k1*z + k0 with k1 = -sc*rstd*dgamma/M, k0 = -sc*dbeta/M - k1*mean
    k1 = -sc * rs * dgamma_r / npix
    k0 = -sc * dbeta_r / npix - k1 * mu
    terms = (sc * gg).abs() + (k1 * z64).abs() + k0.abs()
    near0 = pre_k.abs() < 1e-6 * (z64 * sc).abs()   # the kernel's fp32 pre-activation may round to either side of 0
    assert_bf16(name + " dz", flat(dz), dz_r, terms, skip=near0)
    assert_f32_sum(name + " dbeta", red0[0], dbeta_r, gg.abs().sum(0))
    assert_f32_sum(name + " dgamma", red0[1], dgamma_r, (gg.abs() * ((z64 - mu).abs() + mu.abs()) * rs).sum(0))


@pytest.mark.parametrize("c,point", BWD_CASES)
def test_bn_act_bwd_fused_instances(cuda_lib, c, point):
    from dasemanticsegmentationaml_b200 import kernels as K
    dy2, u_want, where = point
    t = fused_thresholds(c)
    npix = {"n2-1": t[2] - 1, "n2": t[2], "n4-1": t[4] - 1, "n4": t[4]}[where]
    u, fold = fused_instance(c, npix, dy2)
    assert u == u_want and fold == (c in FOLD_C)
    act = (BWD_C.index(c) + BWD_POINTS.index(point)) % 3
    slope = 0.2
    view = where == "n2"
    g = torch.Generator(device=DEV).manual_seed(c * 131 + npix)
    z, d1, d2, dz, dzbuf, dz_off, gamma, beta, coeff = bwd_inputs(g, c, npix, dy2, view)
    red = torch.zeros(1 + K.BN_RED_REPLICAS, 2, c, device=DEV)
    K.bn_act_bwd_fused(d1, d2, z, dz, coeff["scale"], coeff["shift"], coeff["mean"], coeff["rstd"], red, act, slope)
    dz_r, dgamma_r, dbeta_r, gg, pre_k = bwd_reference(z, d1, d2, gamma, beta, coeff, act, slope)
    name = "bwd_fused %s npix%d act%d" % (_bwd_id(c, point), npix, act)
    print("INSTANCE %s: dy2=%d U=%d fold=%d npix=%d" % (name, dy2, u, fold, npix))
    check_bwd(name, z, dz, red[0], coeff, (dz_r, dgamma_r, dbeta_r), gg, pre_k, npix)
    if view:
        assert_outside_untouched(name, dzbuf, dz_off, c)


@pytest.mark.parametrize("c,npix,dy2,act", [(24, 5003, True, 2), (128, 20000, False, 1), (2048, 77, True, 0),
                                            (40, 3, False, 2)])
def test_bn_act_bwd_two_launch_path(cuda_lib, c, npix, dy2, act):
    """bn_act_bwd_reduce + bn_act_bwd_apply against the same reference, and against the fused launch."""
    from dasemanticsegmentationaml_b200 import kernels as K
    slope = 0.2
    g = torch.Generator(device=DEV).manual_seed(c + npix)
    z, d1, d2, dz, dzbuf, dz_off, gamma, beta, coeff = bwd_inputs(g, c, npix, dy2, True)
    args = (coeff["scale"], coeff["shift"], coeff["mean"], coeff["rstd"])
    red = torch.zeros(2, c, device=DEV)
    K.bn_act_bwd_reduce(d1, d2, z, *args, act, slope, red)
    K.bn_act_bwd_apply(d1, d2, z, dz, *args, red, act, slope)
    dz_r, dgamma_r, dbeta_r, gg, pre_k = bwd_reference(z, d1, d2, gamma, beta, coeff, act, slope)
    name = "bwd_two_launch C%d npix%d" % (c, npix)
    check_bwd(name, z, dz, red, coeff, (dz_r, dgamma_r, dbeta_r), gg, pre_k, npix)
    assert_outside_untouched(name, dzbuf, dz_off, c)
    red_f = torch.zeros(1 + K.BN_RED_REPLICAS, 2, c, device=DEV)
    dzf = torch.empty_like(dz)
    K.bn_act_bwd_fused(d1, d2, z, dzf, *args, red_f, act, slope)
    check_bwd(name + " fused", z, dzf, red_f[0], coeff, (dz_r, dgamma_r, dbeta_r), gg, pre_k, npix)


@pytest.mark.parametrize("c,act,dy2,with_bias", [(24, 2, True, True), (64, 1, False, True), (512, 2, False, False),
                                                 (2048, 1, True, True)])
def test_act_bwd_bias(cuda_lib, c, act, dy2, with_bias):
    from dasemanticsegmentationaml_b200 import kernels as K
    npix, slope = 4133, 0.2
    g = torch.Generator(device=DEV).manual_seed(c + act)
    _, a = rand_view(g, npix, c, c + 8, 8)
    _, d1 = rand_view(g, npix, c, c + 16, 16)
    d2 = rand_view(g, npix, c)[1] if dy2 else None
    dzbuf, dz = nhwc(npix, c, c + 8, 0)
    dbias = torch.randn(c, device=DEV, generator=g) if with_bias else None
    db0 = dbias.clone() if with_bias else None
    K.act_bwd_bias(d1, d2, a, dz, act, slope, dbias)
    a64 = flat(a).double()
    dy = flat(d1).double() + (flat(d2).double() if dy2 else 0.0)
    want = dy * act_mask_grad(a64, act, slope)
    assert_bf16("act_bwd_bias C%d dz" % c, flat(dz), want)
    assert_outside_untouched("act_bwd_bias", dzbuf, 0, c)
    if with_bias:
        assert_f32_sum("act_bwd_bias C%d dbias" % c, dbias, db0.double() + want.sum(0),
                       db0.double().abs() + want.abs().sum(0))
        K.act_bwd_bias(d1, d2, a, dz, act, slope, dbias)   # accumulates
        assert_f32_sum("act_bwd_bias C%d dbias twice" % c, dbias, db0.double() + 2 * want.sum(0),
                       db0.double().abs() + 2 * want.abs().sum(0))


# ------------------------------------------------------------------ variance cancellation
def test_variance_cancellation(cuda_lib):
    """channel_stats + bn_norm_act compute var = E[x^2] - mean^2 in fp32, which loses precision when |mean| >> std.
    Gate: rstd within 1e-3 (relative) at |mean| / std = 8; 32 and 128 are printed, not gated."""
    from dasemanticsegmentationaml_b200 import kernels as K
    c, npix = 64, 1 << 20
    g = torch.Generator(device=DEV).manual_seed(5)
    sign = torch.where(torch.rand(c, device=DEV, generator=g) < 0.5, -1.0, 1.0)
    std = torch.rand(c, device=DEV, generator=g) + 0.5
    worst = {}
    for ratio in (8, 32, 128):
        x = (torch.randn(1, 1, npix, c, device=DEV, generator=g) + ratio * sign) * std
        x = x.to(BF)
        stats = torch.zeros(2, c, device=DEV)
        K.channel_stats(x, stats)
        y = torch.empty_like(x)
        scale, shift, mean, rstd = (torch.empty(c, device=DEV) for _ in range(4))
        K.bn_norm_act(x, y, stats, float(npix), None, None, None, None, True, 0, 0.0, scale, shift, mean, rstd)
        x64 = flat(x).double()
        rstd_r = 1.0 / torch.sqrt(x64.var(0, unbiased=False) + EPS)
        rel = ((rstd.double() - rstd_r).abs() / rstd_r).max().item()
        worst[ratio] = rel
        print("VARIANCE |mean|/std=%d C=%d npix=%d: max rstd relative error %.3e" % (ratio, c, npix, rel))
    assert worst[8] < 1e-3, worst
