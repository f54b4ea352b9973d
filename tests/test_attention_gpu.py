"""Global-pool attention kernels of csrc/attention.cu called directly against float64 references on the same
bf16-rounded inputs: the pooled sums, the tiny dense layers (Linear -> BatchNorm over the batch -> act) and their
backward, and the nearest-neighbour broadcast scale/add with its footprint-sum backward.  Element-wise gates as in
test_norm_gpu (tests/helpers.py)."""
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


def nhwc(n, h, w, c, ld=None, off=0, g=None):
    """(buffer [n, h, w, ld], its channel slice [off, off + c)); random bf16 in the slice when g is given."""
    ld = ld or c
    buf = torch.full((n, h, w, ld), SENTINEL, device=DEV, dtype=BF)
    v = buf[..., off:off + c]
    if g is not None:
        v.copy_(torch.randn(n, h, w, c, device=DEV, generator=g).to(BF))
    return buf, v


def assert_outside_untouched(name, buf, off, c):
    outside = torch.ones(buf.shape[-1], dtype=torch.bool, device=DEV)
    outside[off:off + c] = False
    assert bool((buf[..., outside].float() == SENTINEL).all()), name + ": wrote outside its channel slice"


# ------------------------------------------------------------------ pool_sum
POOL_CASES = [
    # n, hw, c, ld
    (8, 1, 2048, 2048),
    (1, 256 * 512, 24, 40),
    (2, 256 * 512, 8, 8),
    (3, 257, 24, 24),
    (8, 4096, 512, 528),
    (2, 1023, 2048, 2064),
    (5, 77, 8, 24),
]


@pytest.mark.parametrize("case", POOL_CASES, ids=lambda c: "N%d-hw%d-C%d-ld%d" % c)
def test_pool_sum(cuda_lib, case):
    from dasemanticsegmentationaml_b200 import kernels as K
    n, hw, c, ld = case
    g = torch.Generator(device=DEV).manual_seed(hw + c)
    _, x = nhwc(n, 1, hw, c, ld, ld - c, g)
    out0 = torch.randn(n, c, device=DEV, generator=g)
    out = out0.clone()
    K.pool_sum(x, out)
    x64 = x.double().reshape(n, hw, c)
    want, terms = x64.sum(1), x64.abs().sum(1)
    assert_f32_sum("pool_sum %s" % (case,), out, out0.double() + want, out0.double().abs() + terms)
    K.pool_sum(x, out)   # accumulates
    assert_f32_sum("pool_sum %s twice" % (case,), out, out0.double() + 2 * want, out0.double().abs() + 2 * terms)


# ------------------------------------------------------------------ fc_small
FC_CASES = [
    # n, cin, co, has_bn, training, act, in_scale, accumulate_din
    (2, 40, 24, True, True, 1, 1.0, False),
    (7, 520, 128, True, True, 3, 1.0 / 49, True),
    (8, 256, 256, False, False, 3, 1.0, False),
    (9, 72, 64, True, False, 1, 0.25, True),
    (33, 1024, 128, True, True, 0, 1.0 / 64, False),
    (64, 136, 40, True, True, 3, 1.0, True),
    (64, 24, 256, False, False, 1, 0.5, True),
    (7, 8, 8, True, False, 0, 1.0, False),
]


def _fc_id(c):
    return "N%d-ci%d-co%d-%s-act%d-s%g%s" % (c[0], c[1], c[2], ("bn_train" if c[4] else "bn_eval") if c[3] else "nobn",
                                             c[5], c[6], "-accdin" if c[7] else "")


@pytest.mark.parametrize("case", FC_CASES, ids=_fc_id)
def test_fc_small(cuda_lib, case):
    from dasemanticsegmentationaml_b200 import kernels as K
    n, cin, co, has_bn, training, act, in_scale, acc_din = case
    g = torch.Generator(device=DEV).manual_seed(n * 1000 + cin + co)
    inp = torch.rand(n, cin, device=DEV, generator=g) * 2.0        # pooled activations
    W = torch.randn(co, cin, device=DEV, generator=g) / cin ** 0.5
    gamma = torch.rand(co, device=DEV, generator=g) + 0.5
    beta = torch.randn(co, device=DEV, generator=g) * 0.5
    rm0 = torch.randn(co, device=DEV, generator=g) * 0.1
    rv0 = torch.rand(co, device=DEV, generator=g) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    pre, out = torch.empty(n, co, device=DEV), torch.empty(n, co, device=DEV)
    mean, rstd = torch.full((co,), float("nan"), device=DEV), torch.full((co,), float("nan"), device=DEV)
    K.fc_small_fwd(inp, in_scale, W, (gamma, beta, rm, rv) if has_bn else None, training, act, pre, out,
                   mean if has_bn else None, rstd if has_bn else None, momentum=MOMENTUM, eps=EPS)

    # float64 reference: Linear, BatchNorm over the batch, act -- forward and autograd backward
    in64 = inp.double().requires_grad_(True)
    W64 = W.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = beta.double().requires_grad_(True)
    pre64 = in_scale * in64 @ W64.t()
    pre64.retain_grad()
    S = abs(in_scale) * inp.double() @ W.double().abs().t()        # sum of |terms| of each pre-activation
    name = "fc_small %s" % _fc_id(case)
    assert_within(name + " pre", pre, pre64.detach(), 1e-5 * S + 1e-6)
    if has_bn:
        if training:
            m64, v64 = pre64.detach().mean(0), pre64.detach().var(0, unbiased=False)
            t64 = F.batch_norm(pre64, None, None, g64, b64, training=True, eps=EPS)
        else:
            m64, v64 = rm0.double(), rv0.double()
            t64 = F.batch_norm(pre64, m64, v64, g64, b64, training=False, eps=EPS)
        rs64 = 1.0 / torch.sqrt(v64 + EPS)
        Sm = S.mean(0)
        assert_within(name + " mean", mean, m64, 1e-5 * Sm + 1e-6)
        assert_within(name + " rstd", rstd, rs64, rs64 * (1e-5 * (1 + Sm * rs64)))
        xh = (pre64.detach() - m64) * rs64
        out_terms = 3 * S * rs64 * g64.detach().abs() + (g64.detach() * xh).abs() + b64.detach().abs()
        if training:
            unb = v64 * n / (n - 1)
            assert_within(name + " running_mean", rm, 0.9 * rm0.double() + 0.1 * m64,
                          1e-5 * (rm0.double().abs() + Sm) + 1e-6)
            assert_within(name + " running_var", rv, 0.9 * rv0.double() + 0.1 * unb,
                          1e-5 * (rv0.double() + unb + 2 * unb.sqrt() * Sm) + 1e-6)
        else:
            assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
    else:
        t64 = pre64
        out_terms = S
    if act == 1:
        want = torch.relu(t64)
    elif act == 3:
        want = torch.sigmoid(t64)
    else:
        want = t64
    assert_within(name + " out", out, want.detach(), 1e-5 * out_terms + 1e-6)

    # backward into non-zero (accumulating) buffers
    dout = torch.randn(n, co, device=DEV, generator=g)
    if act == 1:
        gg = dout.double() * (out > 0).double()                   # the kernel's mask: its own forward output
    elif act == 3:
        s = torch.sigmoid(t64.detach())
        gg = dout.double() * s * (1 - s)
    else:
        gg = dout.double()
    t64.backward(gg)
    dW0 = torch.randn(co, cin, device=DEV, generator=g)
    dg0, db0 = torch.randn(co, device=DEV, generator=g), torch.randn(co, device=DEV, generator=g)
    din0 = torch.randn(n, cin, device=DEV, generator=g)
    dW, dgamma, dbeta, din = dW0.clone(), dg0.clone(), db0.clone(), din0.clone()
    scratch = torch.empty(n, co, device=DEV)
    K.fc_small_bwd(dout, out, pre, inp, in_scale, W, has_bn, training, gamma if has_bn else None,
                   mean if has_bn else None, rstd if has_bn else None, act, scratch, dW,
                   dgamma if has_bn else None, dbeta if has_bn else None, din, accumulate_din=acc_din)
    if has_bn:
        A = (gamma.double() * rs64).abs() * (gg.abs() + (gg.abs().mean(0) + xh.abs() * (gg * xh).abs().mean(0)
                                                          if training else 0.0))
        assert_f32_sum(name + " dbeta", dbeta, db0.double() + b64.grad, db0.double().abs() + gg.abs().sum(0))
        assert_f32_sum(name + " dgamma", dgamma, dg0.double() + g64.grad, dg0.double().abs() + (gg * xh).abs().sum(0))
    else:
        A = gg.abs()
        assert torch.equal(dgamma, dg0) and torch.equal(dbeta, db0)
    assert_f32_sum(name + " dpre", scratch, pre64.grad, A)
    assert_f32_sum(name + " dW", dW, dW0.double() + W64.grad, dW0.double().abs() + abs(in_scale) * A.t() @ inp.double())
    din_want = in64.grad + (din0.double() if acc_din else 0.0)
    din_terms = abs(in_scale) * A @ W.double().abs() + (din0.double().abs() if acc_din else 0.0)
    assert_f32_sum(name + " din", din, din_want, din_terms)


def test_fc_small_refuses_batches_over_64(cuda_lib):
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200._lib import B200Error
    n, cin, co = 65, 32, 16
    inp, W = torch.rand(n, cin, device=DEV), torch.randn(co, cin, device=DEV)
    pre, out = torch.full((n, co), 3.0, device=DEV), torch.full((n, co), 3.0, device=DEV)
    with pytest.raises(B200Error, match=r"\(-1\)"):
        K.fc_small_fwd(inp, 1.0, W, None, False, 0, pre, out, None, None)
    scratch, dW, din = torch.empty(n, co, device=DEV), torch.zeros(co, cin, device=DEV), torch.zeros(n, cin, device=DEV)
    with pytest.raises(B200Error, match=r"\(-1\)"):
        K.fc_small_bwd(out, out, pre, inp, 1.0, W, False, False, None, None, None, 0, scratch, dW, None, None, din)
    torch.cuda.synchronize()
    assert bool((out == 3.0).all()) and bool((dW == 0).all())


# ------------------------------------------------------------------ nearest broadcast scale/add and its backward
SIZE_PAIRS = [
    ((16, 24), (16, 24)),    # identity
    ((8, 12), (16, 24)),     # exactly 2x
    ((8, 12), (15, 23)),     # 2h - 1
    ((23, 7), (45, 64)),     # non-integer up-sampling
    ((45, 45), (23, 23)),    # down-sampling: source pixels with an empty footprint
    ((23, 45), (45, 23)),    # up along h, down along w
]
# which optional operands are given: forward (s, v, t), backward (dsum, b -> dot, vsum)
VARIANTS = [dict(s=1, v=1, t=1, dsum=1, b=1, vsum=1), dict(s=0, v=0, t=0, dsum=0, b=1, vsum=0),
            dict(s=1, v=0, t=1, dsum=1, b=0, vsum=1), dict(s=0, v=1, t=0, dsum=1, b=1, vsum=0)]
BCAST_CASES = [pytest.param(sp, vi, c, id="%dx%d-%dx%d-v%d-C%d" % (sp[0] + sp[1] + (vi, c)))
               for i, sp in enumerate(SIZE_PAIRS) for vi in range(len(VARIANTS)) for c in ((24,) if (i + vi) % 2 else (64,))]


def nearest(x64, ho, wo):
    """F.interpolate(mode="nearest") of an NHWC float64 tensor."""
    return F.interpolate(x64.permute(0, 3, 1, 2), size=(ho, wo), mode="nearest").permute(0, 2, 3, 1)


@pytest.mark.parametrize("sizes,variant,c", BCAST_CASES)
def test_scale_add_bcast(cuda_lib, sizes, variant, c):
    from dasemanticsegmentationaml_b200 import kernels as K
    (hs, ws), (ho, wo) = sizes
    opt = VARIANTS[variant]
    n = 2
    g = torch.Generator(device=DEV).manual_seed(hs * ws + ho * wo + variant)
    _, a = nhwc(n, hs, ws, c, c + 8, 8, g)
    s = torch.rand(n, c, device=DEV, generator=g) if opt["s"] else None
    v = torch.randn(n, c, device=DEV, generator=g) if opt["v"] else None
    t = nhwc(n, hs, ws, c, c + 16, 0, g)[1] if opt["t"] else None
    s_plus, v_scale = 0.75, 1.5
    obuf, out = nhwc(n, ho, wo, c, c + 24, 16)
    K.scale_add_bcast(a, s, s_plus, v, v_scale, t, out)
    A = nearest(a.double(), ho, wo)
    sv = (s.double() if s is not None else torch.zeros(n, c, device=DEV, dtype=F64))[:, None, None, :] + s_plus
    want = A * sv
    terms = (A * sv).abs()
    if v is not None:
        want = want + (v.double() * v_scale)[:, None, None, :]
        terms = terms + (v.double() * v_scale).abs()[:, None, None, :]
    if t is not None:
        T = nearest(t.double(), ho, wo)
        want, terms = want + T, terms + T.abs()
    name = "scale_add_bcast %dx%d->%dx%d C%d %s" % (hs, ws, ho, wo, c, opt)
    assert_bf16(name, out, want, terms)
    assert_outside_untouched(name, obuf, 16, c)


@pytest.mark.parametrize("sizes,variant,c", BCAST_CASES)
def test_upsum_dot_reduce(cuda_lib, sizes, variant, c):
    from dasemanticsegmentationaml_b200 import kernels as K
    (hs, ws), (ho, wo) = sizes
    opt = VARIANTS[variant]
    n = 2
    g = torch.Generator(device=DEV).manual_seed(hs * ws + ho * wo + variant + 1)
    _, dout = nhwc(n, ho, wo, c, c + 8, 0, g)
    b = nhwc(n, hs, ws, c, c + 16, 8, g)[1] if opt["b"] else None
    dbuf, dsum = nhwc(n, hs, ws, c, c + 24, 16) if opt["dsum"] else (None, None)
    dot0, vsum0 = torch.randn(n, c, device=DEV, generator=g), torch.randn(n, c, device=DEV, generator=g)
    dot, vsum = dot0.clone(), (vsum0.clone() if opt["vsum"] else None)
    K.upsum_dot_reduce(dout, b, dsum, hs, ws, dot, vsum)

    def footprint_sum(d64):   # autograd backward of the nearest up-sampling: the footprint sum per source pixel
        src = torch.zeros(n, hs, ws, c, device=DEV, dtype=F64, requires_grad=True)
        nearest(src, ho, wo).backward(d64)
        return src.grad

    ds = footprint_sum(dout.double())
    ds_abs = footprint_sum(dout.double().abs())
    name = "upsum_dot_reduce %dx%d->%dx%d C%d %s" % (ho, wo, hs, ws, c, opt)
    if dsum is not None:
        assert_bf16(name + " dsum", dsum, ds, ds_abs)
        assert_outside_untouched(name, dbuf, 16, c)
    if b is not None:
        b64 = b.double()
        assert_f32_sum(name + " dot", dot, dot0.double() + (ds * b64).sum((1, 2)),
                       dot0.double().abs() + (ds_abs * b64.abs()).sum((1, 2)))
    else:
        assert torch.equal(dot, dot0)
    if vsum is not None:
        assert_f32_sum(name + " vsum", vsum, vsum0.double() + ds.sum((1, 2)), vsum0.double().abs() + ds_abs.sum((1, 2)))
