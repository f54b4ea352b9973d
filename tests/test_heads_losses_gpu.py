"""The discriminator classifier (csrc/classifier.cu), the stem unfold (csrc/stem.cu) and the loss helpers of
csrc/loss.cu called directly: against float64 references on the same inputs, bit-exact where the operation is
exact (stem_im2col, cast_f32_bf16, radix_select_desc).  Element-wise gates as in test_norm_gpu (tests/helpers.py)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import assert_bf16, assert_f32_sum, assert_within, rel_l2

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64
DEV = "cuda"
SENTINEL = -7.0


def nchw(t):
    return t.permute(0, 3, 1, 2)


# ------------------------------------------------------------------ classifier Conv2d(C, 1, 4, 2, 1)
CLS_CASES = [(2, 11, 19, 64), (8, 3, 5, 512), (1, 11, 19, 1024), (3, 3, 5, 64), (8, 11, 19, 512), (4, 2, 3, 64)]


@pytest.mark.parametrize("case", CLS_CASES, ids=lambda c: "N%d-%dx%d-C%d" % c)
def test_classifier(cuda_lib, case):
    from dasemanticsegmentationaml_b200 import kernels as K
    n, h, w, c = case
    ho, wo = (h + 2 - 4) // 2 + 1, (w + 2 - 4) // 2 + 1
    g = torch.Generator(device=DEV).manual_seed(n * h * w + c)
    xbuf = torch.full((n, h, w, c + 16), SENTINEL, device=DEV, dtype=BF)
    x = xbuf[..., 8:8 + c]
    x.copy_(torch.randn(n, h, w, c, device=DEV, generator=g).to(BF))
    wt = torch.randn(1, c, 4, 4, device=DEV, generator=g) / (4 * c ** 0.5)
    bias = torch.randn(1, device=DEV, generator=g)
    name = "classifier N%d %dx%d C%d" % case

    out = torch.full((n, ho, wo), float("nan"), device=DEV)
    K.classifier_fwd(x, wt, bias, out)
    x64 = nchw(x.double()).contiguous().requires_grad_(True)
    w64 = wt.double().requires_grad_(True)
    b64 = bias.double().requires_grad_(True)
    ref = F.conv2d(x64, w64, b64, stride=2, padding=1)
    terms = F.conv2d(nchw(x.double()).abs(), wt.double().abs(), stride=2, padding=1) + bias.double().abs()
    assert_f32_sum(name + " fwd", out, ref.detach()[:, 0], terms[:, 0])

    dout = torch.randn(n, ho, wo, device=DEV, generator=g)
    ref.backward(dout.double()[:, None])
    xa = nchw(x.double()).abs().contiguous().requires_grad_(True)
    wa = wt.double().abs().requires_grad_(True)
    F.conv2d(xa, wa, stride=2, padding=1).backward(dout.double().abs()[:, None])

    dxbuf = torch.full((n, h, w, c + 24), SENTINEL, device=DEV, dtype=BF)
    dx = dxbuf[..., 16:16 + c]
    K.classifier_dgrad(dout, wt, dx)
    assert_bf16(name + " dgrad", dx, x64.grad.permute(0, 2, 3, 1), xa.grad.permute(0, 2, 3, 1))
    assert bool((dxbuf[..., :16].float() == SENTINEL).all() and (dxbuf[..., 16 + c:].float() == SENTINEL).all())

    dw0, db0 = torch.randn(1, c, 4, 4, device=DEV, generator=g), torch.randn(1, device=DEV, generator=g)
    dw, db = dw0.clone(), db0.clone()
    K.classifier_wgrad(dout, x, dw, db)   # accumulates into dw, dbias
    assert_f32_sum(name + " dw", dw, dw0.double() + w64.grad, dw0.double().abs() + wa.grad)
    assert_f32_sum(name + " dbias", db, db0.double() + b64.grad, db0.double().abs() + dout.double().abs().sum())


# ------------------------------------------------------------------ stem unfold
@pytest.mark.parametrize("n,h,w,col_ld", [(2, 37, 61, 48), (1, 64, 33, 32), (3, 1, 5, 40), (1, 9, 2, 64)])
def test_stem_im2col_bit_exact(cuda_lib, n, h, w, col_ld):
    from dasemanticsegmentationaml_b200 import kernels as K
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    g = torch.Generator(device=DEV).manual_seed(h * w)
    img = torch.randn(n, 3, h, w, device=DEV, generator=g)
    buf = torch.full((n, ho, wo, col_ld), SENTINEL, device=DEV, dtype=BF)
    K.stem_im2col(img, buf[..., :32])
    want = F.unfold(img, 3, padding=1, stride=2).reshape(n, 27, ho, wo).permute(0, 2, 3, 1).to(BF)
    assert torch.equal(buf[..., :27].contiguous().view(torch.int16), want.contiguous().view(torch.int16))
    assert torch.equal(buf[..., 27:32].contiguous().view(torch.int16), torch.zeros(n, ho, wo, 5, device=DEV, dtype=torch.int16))
    assert bool((buf[..., 32:].float() == SENTINEL).all())


# ------------------------------------------------------------------ BCE-with-logits against a constant target
@pytest.mark.parametrize("count", [1, 7, 1000, 1 << 20])
@pytest.mark.parametrize("target", [0.0, 1.0])
def test_bce_const(cuda_lib, count, target):
    from dasemanticsegmentationaml_b200 import kernels as K
    g = torch.Generator(device=DEV).manual_seed(count)
    x = torch.randn(count, device=DEV, generator=g) * 8
    special = torch.tensor([100.0, -100.0, 0.0, 30.0, -30.0], device=DEV)
    x[:min(count, 5)] = special[:min(count, 5)]
    x64 = x.double()
    loss_terms = x64.clamp_min(0) + (x64 * target).abs() + torch.log1p(torch.exp(-x64.abs()))
    want = F.binary_cross_entropy_with_logits(x64, torch.full_like(x64, target))
    out = torch.full((1,), 0.25, device=DEV)
    K.bce_const_fwd(x, target, out)                     # out[0] += mean loss
    assert_f32_sum("bce_fwd n%d t%g" % (count, target), out[0], 0.25 + want, 0.25 + loss_terms.mean())
    sig = torch.sigmoid(x64)
    for gscale in (None, torch.tensor([0.37], device=DEV)):
        gmul = 2.0
        gs = (1.0 if gscale is None else gscale.double()) * gmul / count
        dx = torch.empty_like(x)
        K.bce_const_bwd(x, target, gscale, gmul, dx)
        want_dx = (sig - target) * gs
        assert_within("bce_bwd n%d t%g gscale=%s" % (count, target, gscale is not None), dx, want_dx,
                      1e-5 * (sig + target) * abs(gs) + 1e-30)


# ------------------------------------------------------------------ radix select + OHEM reduction
def loss_like(kind, count, g):
    if kind == "random":
        x = torch.rand(count, device=DEV, generator=g) * 5
    elif kind == "ties":
        x = torch.randint(0, 6, (count,), device=DEV, generator=g).float() * 0.375
    elif kind == "all_equal":
        x = torch.full((count,), 1.25, device=DEV)
    else:   # "zeros": more than half exact zeros, like the loss map of ignored pixels
        x = torch.rand(count, device=DEV, generator=g) * 3
        x[torch.rand(count, device=DEV, generator=g) < 0.6] = 0.0
    return x


@pytest.mark.parametrize("kind", ["random", "ties", "all_equal", "zeros"])
@pytest.mark.parametrize("count", [1, 1000, 1 << 20])
def test_radix_select_desc_bit_exact(cuda_lib, kind, count):
    from dasemanticsegmentationaml_b200 import kernels as K
    g = torch.Generator(device=DEV).manual_seed(count + len(kind))
    x = loss_like(kind, count, g)
    desc = np.sort(x.cpu().numpy())[::-1]
    state = torch.empty(2, dtype=torch.int32, device=DEV)
    hist = torch.empty(256, dtype=torch.int32, device=DEV)
    for rank in sorted({0, count // 3, count // 2, count - 1}):
        K.radix_select_desc(x, rank, state, hist)
        got = state[:1].view(torch.float32).item()
        assert np.float32(got).tobytes() == desc[rank].tobytes(), (kind, count, rank, got, desc[rank])


def ohem_reference(x64, threshold, keep):
    """OHEM_CrossEntroy_Loss's sort formulation (oracle.segnet_oracle.ohem_cross_entropy) on a loss map, with the
    per-element gradient from autograd."""
    xr = x64.clone().requires_grad_(True)
    s, _ = torch.sort(xr, descending=True)
    loss = s[s > threshold].mean() if s[keep] > threshold else s[:keep].mean()
    loss.backward()
    return loss.detach(), xr.grad, s[keep].item()


@pytest.mark.parametrize("kind,threshold,keep_frac", [("random", 0.3567, 0.001), ("random", 4.9, 0.3),
                                                      ("ties", 0.1, 0.5), ("ties", 2.0, 0.2),
                                                      ("zeros", 0.3567, 0.7), ("zeros", 0.3567, 0.0001),
                                                      ("all_equal", 0.3567, 0.5)])
def test_ohem_reduce_and_weights(cuda_lib, kind, threshold, keep_frac):
    from dasemanticsegmentationaml_b200 import kernels as K
    count = 300007
    keep = int(keep_frac * count)
    g = torch.Generator(device=DEV).manual_seed(count + keep)
    x = loss_like(kind, count, g)
    state = torch.empty(2, dtype=torch.int32, device=DEV)
    hist = torch.empty(256, dtype=torch.int32, device=DEV)
    K.radix_select_desc(x, keep, state, hist)
    sums = torch.empty(5, dtype=F64, device=DEV)
    sel = torch.empty(4, dtype=torch.float32, device=DEV)
    K.ohem_reduce(x, state, threshold, keep, sums, sel)
    wts = torch.empty_like(x)
    K.ohem_weights(x, sel, wts)
    x64 = x.double()
    loss, grad, cut = ohem_reference(x64, threshold, keep)
    name = "ohem %s thr%g keep%d" % (kind, threshold, keep)
    assert_within(name + " loss", sel[0], loss, 1e-6 * loss.abs() + 1e-30)
    if cut > threshold:
        assert sel[1].item() == np.float32(threshold)
        assert_within(name + " weights", wts, grad, 1e-6 * grad.abs() + 1e-30)
    else:
        # a cut inside a run of ties: the kernel spreads the remaining weight evenly over the tied elements, sort
        # gives it to some of them -- the same loss, and the same total weight on the run
        assert sel[1].item() == np.float32(cut)
        tie = x64 == cut
        print("%s: cut %.4f, %d tied elements" % (name, cut, int(tie.sum())))
        assert_within(name + " weights off the cut", wts[~tie], grad[~tie], 1e-6 * grad[~tie].abs() + 1e-30)
        assert bool((wts[tie] == wts[tie][0]).all())
        assert_within(name + " weight on the cut", wts[tie].double().sum(), grad[tie].sum(), 1e-6 * grad[tie].sum() + 1e-12)


def test_ohem_with_ignored_pixels_end_to_end(cuda_lib):
    """upsample_ohem_cross_entropy with labels holding 255 (the ignored pixels of a Cityscapes / GTA5 label map)
    against the oracle's sort formulation.  Such pixels contribute a zero loss and no gradient; the oracle's
    F.cross_entropy does the same for its own ignore index, -100.  With more than half the pixels ignored, the
    second keep_num lands in the run of zero losses."""
    from dasemanticsegmentationaml_b200 import losses as L
    from oracle import segnet_oracle as O
    n, h, w, H, W = 2, 16, 32, 128, 256
    g = torch.Generator().manual_seed(19)
    lr = torch.zeros(n, h, w, 32)
    lr[..., :19] = 3 * torch.randn(n, h, w, 19, generator=g)
    lr = lr.to(DEV)
    labels = torch.randint(0, 19, (n, H, W), generator=g)
    labels[torch.rand(n, H, W, generator=g) < 0.55] = 255
    labels = labels.to(DEV)
    for thr, keep in ((0.3567, 1000), (0.3567, int(0.7 * n * H * W))):
        a = lr.clone().requires_grad_(True)
        b = lr.double().requires_grad_(True)
        v1 = L.upsample_ohem_cross_entropy(a, labels, thr, keep)
        full = F.interpolate(nchw(b[..., :19]), (H, W), mode="bilinear", align_corners=True)
        v2 = O.ohem_cross_entropy(full, labels.masked_fill(labels == 255, -100), thr, keep)
        assert abs(v1.item() - v2.item()) < 1e-5 * abs(v2.item()), (thr, keep, v1.item(), v2.item())
        v1.backward()
        v2.backward()
        assert rel_l2(a.grad, b.grad) < 1e-4, (thr, keep)


# ------------------------------------------------------------------ fp32 -> bf16 cast, fp32 scale
def special_f32():
    """fp32 bit patterns where a conversion goes wrong: exact ties between two bf16 values (both parities),
    +-inf, NaN, denormals (tie and non-tie), values that round up past the largest bf16 to inf."""
    bits = []
    for hi in (0x3F80, 0x3F81, 0xBF80, 0xBF81, 0x0001, 0x0002, 0x007F, 0x8001, 0x7F7E, 0x7F7F, 0xFF7F):
        for lo in (0x0000, 0x7FFF, 0x8000, 0x8001, 0xFFFF):
            bits.append((hi << 16) | lo)
    bits += [0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001, 0x00000001, 0x80000001, 0x007FFFFF,
             0x00008000, 0x00018000, 0x7F7FFFFF, 0x80000000, 0x00000000]
    while len(bits) % 4:
        bits.append(0x3F800000)
    return torch.tensor(np.array(bits, dtype=np.uint32).view(np.int32)).view(torch.float32)


def test_cast_f32_bf16_bit_exact(cuda_lib):
    from dasemanticsegmentationaml_b200 import kernels as K
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.cat([special_f32().to(DEV), torch.randn(1 << 16, device=DEV, generator=g) * 100,
                   torch.randn(4096, device=DEV, generator=g) * 1e-39])
    y = torch.full(x.shape, SENTINEL, device=DEV, dtype=BF)
    K.cast_f32_bf16(x, y)
    want = x.cpu().to(BF).to(DEV)
    nan = torch.isnan(want)
    assert bool((torch.isnan(y) == nan).all())
    assert torch.equal(y[~nan].view(torch.int16), want[~nan].view(torch.int16))


@pytest.mark.parametrize("with_den", [False, True])
def test_scale_f32(cuda_lib, with_den):
    from dasemanticsegmentationaml_b200 import kernels as K
    g = torch.Generator(device=DEV).manual_seed(4)
    x = torch.cat([special_f32().to(DEV), torch.randn(1 << 16, device=DEV, generator=g) * 100,
                   torch.tensor([3e38, -3e38, 1e-30, 2.5e-38], device=DEV)])
    num = torch.tensor([3.5], device=DEV)
    den = torch.tensor([1.75e3 if with_den else 0.0], device=DEV, dtype=F64)
    mul = 2.0
    y = torch.empty_like(x)
    K.scale_f32(x, num, den if with_den else None, mul, y)
    want = x.double() * 3.5 * mul / (den.item() if with_den else 1.0)
    want32 = want.float()
    nan = torch.isnan(want32)
    assert bool((torch.isnan(y) == nan).all())
    inf = torch.isinf(want32)
    assert torch.equal(y[inf], want32[inf])          # overflow to inf and inf inputs keep their sign
    fin = ~nan & ~inf
    # loss.cu is compiled flush-to-zero (build.py): a denormal input or a result below the smallest normal float
    # may come out as a zero of the same sign; everything else within a few fp32 ulp of the float64 value
    tiny = (want[fin].abs() < 2.0 ** -126) | (x[fin].abs() < 2.0 ** -126)
    flushed = tiny & (y[fin] == 0) & (torch.signbit(y[fin]) == torch.signbit(want32[fin]))
    assert_within("scale_f32 den=%s" % with_den, y[fin], want[fin], 6e-7 * want[fin].abs() + 2.0 ** -149, skip=flushed)
