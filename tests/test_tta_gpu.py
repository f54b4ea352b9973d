"""Multi-scale + flip evaluation (BiSeNet's MscEval), from the csrc/msc.cu kernels up to train.predict / val.

Kernel level: image_rescale against torch's fp32 F.interpolate(align_corners=True) and torch.flip;
msc_argmax against a float64 softmax sum over the same fp32 logit maps (NaN padding classes, tight and
32-float pixel strides, mirrored halves passed as offset views of a 2N buffer).

Model level: train.predict against the fp32 restatement of MscEval below (msc_predict, built from the
oracle's bisenet_lowres), with the argmax-agreement gate of tests/test_modules_gpu.py, and the default
single-scale path of eval_batch / val against the code it replaced."""
import pytest
import torch
import torch.nn.functional as F

from oracle import segnet_oracle as O
from tests.helpers import load_oracle_state, to_device

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64 = torch.float64
GAP = 1e-4   # top-two gap (summed probabilities) above which the prediction must be exact


def _round4(n):
    return (n + 3) // 4 * 4


def msc_predict(sd, images, n_classes, scales, flip):
    """BiSeNet's MscEval(scales, flip) over the oracle network: for each scale the images resized to
    (int(s*H), int(s*W)) (bilinear, align_corners=True), and with flip their mirrors; each run's `out` logits
    up-sampled to H x W, mirrored runs flipped back, softmax summed in fp32.  Returns (argmax, the sum)."""
    _, _, H, W = images.shape
    total = None
    for s in scales:
        xs = F.interpolate(images, (int(s * H), int(s * W)), mode="bilinear", align_corners=True)
        runs = [(xs, False)] + ([(torch.flip(xs, dims=[3]), True)] if flip else [])
        for x, mirrored in runs:
            out = O.bisenet_lowres(sd, x, training=False)[0][:, :n_classes]
            up = F.interpolate(out, (H, W), mode="bilinear", align_corners=True)
            if mirrored:
                up = torch.flip(up, dims=[3])
            p = torch.softmax(up.float(), dim=1)
            total = p if total is None else total + p
    return total.argmax(1), total


def _gap(prob_sum):
    top = prob_sum.topk(2, dim=1).values
    return top[:, 0] - top[:, 1]


def _assert_argmax(name, pred, ref_sum):
    """Exact wherever the float64 top-two gap exceeds GAP, and equal on >= 99.9 % of all pixels."""
    ref = ref_sum.argmax(1)
    clear = _gap(ref_sum) > GAP
    wrong = int(((pred.long() != ref) & clear).sum())
    agree = (pred.long() == ref).double().mean().item()
    print("%s: %d clear-gap mismatches, agreement %.6f" % (name, wrong, agree))
    assert wrong == 0, name
    assert agree >= 0.999, (name, agree)


# ------------------------------------------------------------------ image_rescale
# (H, W, h, w): down- and up-scaling of 512x1024 at 0.5 / 0.75 / 1.25 / 1.75, Cityscapes' 720x1280 at 0.75,
# an odd size, and the identity (an exact copy)
RESCALE_CASES = [(512, 1024, 256, 512), (512, 1024, 384, 768), (512, 1024, 640, 1280), (512, 1024, 896, 1792),
                 (720, 1280, 540, 960), (37, 53, 64, 91), (512, 1024, 512, 1024)]


@pytest.mark.parametrize("case", RESCALE_CASES, ids=["%dx%d-%dx%d" % c for c in RESCALE_CASES])
def test_image_rescale_against_torch(cuda_lib, case):
    from dasemanticsegmentationaml_b200 import kernels as K
    H, W, h, w = case
    n = 3
    x = torch.randn(n, 3, H, W, generator=torch.Generator().manual_seed(H + w)).to(DEV)
    ref = F.interpolate(x, (h, w), mode="bilinear", align_corners=True)
    for mirror in (False, True):
        dst = torch.full((n * (2 if mirror else 1), 3, h, w), float("nan"), device=DEV)
        K.image_rescale(x, dst, mirror=mirror)
        err = (dst[:n] - ref).abs().max().item()
        print("rescale %s mirror=%d max|d| %.3g" % (case, mirror, err))
        assert err <= 1e-5
        if mirror:
            assert torch.equal(dst[n:], torch.flip(dst[:n], dims=[3]))
        if (h, w) == (H, W):
            assert torch.equal(dst[:n], x)


def test_image_rescale_refuses_malformed(cuda_lib):
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200._lib import B200Error
    x = torch.randn(33, 3, 16, 16, device=DEV)
    K.image_rescale(x, torch.empty(33, 3, 8, 8, device=DEV))                 # 33 images without mirrors run
    with pytest.raises(B200Error, match="batch limit"):
        K.image_rescale(x, torch.empty(66, 3, 8, 8, device=DEV), mirror=True)
    with pytest.raises(B200Error, match="positive"):
        K.image_rescale(x[:2], torch.empty(2, 3, 0, 8, device=DEV))
    torch.cuda.synchronize()


# ------------------------------------------------------------------ msc_argmax
MAP_SIZES = [(16, 32), (23, 40), (12, 20), (9, 17), (30, 61)]
OUT_HW = (128, 240)


def _maps(n_maps, n_classes, ld, n, seed):
    """fp32 NHWC maps with NaN padding classes; every odd map is mirrored and passed as the second half of a
    2N buffer.  Returns (views for the kernel, mirrored flags, float64 softmax sum)."""
    g = torch.Generator().manual_seed(seed)
    H, W = OUT_HW
    views, flags, total = [], [], torch.zeros(n, n_classes, H, W, dtype=F64, device=DEV)
    for k in range(n_maps):
        h, w = MAP_SIZES[k % len(MAP_SIZES)]
        mirrored = k % 2 == 1
        buf = torch.full((2 * n if mirrored else n, h, w, ld), float("nan"))
        buf[..., :n_classes] = 3 * torch.randn(buf.shape[:3] + (n_classes,), generator=g)
        buf = buf.to(DEV)
        view = buf[n:] if mirrored else buf
        up = F.interpolate(view[..., :n_classes].double().permute(0, 3, 1, 2), (H, W), mode="bilinear",
                           align_corners=True)
        if mirrored:
            up = torch.flip(up, dims=[3])
        total += torch.softmax(up, dim=1)
        views.append(view)
        flags.append(mirrored)
    return views, flags, total


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64], ids=["u8", "i64"])
@pytest.mark.parametrize("ld_kind", ["tight", "32"])
@pytest.mark.parametrize("n_classes", [2, 3, 13, 16, 19, 24, 32])
@pytest.mark.parametrize("n_maps", [1, 2, 5, 12, 16])
def test_msc_argmax_against_float64(cuda_lib, n_maps, n_classes, ld_kind, dtype):
    from dasemanticsegmentationaml_b200 import kernels as K
    ld = _round4(n_classes) if ld_kind == "tight" else 32
    n = 1 + n_maps % 3
    views, flags, ref_sum = _maps(n_maps, n_classes, ld, n, seed=1000 * n_maps + n_classes)
    if n_maps == 1:   # one map: also run it mirrored
        flags = [True]
        ref_sum = torch.softmax(torch.flip(F.interpolate(views[0][..., :n_classes].double().permute(0, 3, 1, 2),
                                                         OUT_HW, mode="bilinear", align_corners=True), dims=[3]), dim=1)
    pred = torch.full((n,) + OUT_HW, 255 if dtype == torch.uint8 else -1, dtype=dtype, device=DEV)
    K.msc_argmax(views, flags, OUT_HW[0], OUT_HW[1], n_classes, pred)
    _assert_argmax("msc_argmax %d maps %d classes ld %d" % (n_maps, n_classes, ld), pred, ref_sum)


def test_msc_argmax_refuses_malformed(cuda_lib):
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200._lib import B200Error
    lr = torch.zeros(1, 8, 8, 32, device=DEV)
    pred = torch.empty(1, 32, 32, dtype=torch.uint8, device=DEV)
    K.msc_argmax([lr] * 16, [False] * 16, 32, 32, 19, pred)
    with pytest.raises(B200Error, match="maps"):
        K.msc_argmax([], [], 32, 32, 19, pred)
    with pytest.raises(B200Error, match="maps"):
        K.msc_argmax([lr] * 17, [False] * 17, 32, 32, 19, pred)
    with pytest.raises(B200Error, match="stride"):
        K.msc_argmax([torch.zeros(1, 8, 8, 30, device=DEV)], [True], 32, 32, 19, pred)
    with pytest.raises(B200Error, match="stride"):
        K.msc_argmax([torch.zeros(1, 8, 8, 16, device=DEV)], [True], 32, 32, 19, pred)
    for bad in (1, 33):
        with pytest.raises(B200Error, match="classes"):
            K.msc_argmax([lr, lr], [False, True], 32, 32, bad, pred)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ the network
@pytest.fixture(scope="module")
def net19(cuda_lib):
    from dasemanticsegmentationaml_b200.model import BiSeNet
    sd = O.make_bisenet_state(seed=0)
    return load_oracle_state(BiSeNet("STDCNet813", 19), sd).to(DEV).eval(), to_device(sd, DEV)


def test_predict_flip_teacher_forced(net19):
    """scales=(1.0,), flip=True: predict against the float64 combine of the model's own two maps."""
    from dasemanticsegmentationaml_b200 import train as T
    m, _ = net19
    x = torch.randn(2, 3, 256, 512, generator=torch.Generator().manual_seed(11)).to(DEV)
    pred = T.predict(m, x, scales=(1.0,), flip=True, pred_dtype=torch.int64)
    assert pred.shape == (2, 256, 512) and pred.dtype == torch.int64
    with torch.no_grad():
        lr = m.forward_lowres(torch.cat([x, torch.flip(x, dims=[3])]))[0]

    def up(t):
        return F.interpolate(t[..., :19].double().permute(0, 3, 1, 2), (256, 512), mode="bilinear", align_corners=True)
    ref_sum = torch.softmax(up(lr[:2]), dim=1) + torch.flip(torch.softmax(up(lr[2:]), dim=1), dims=[3])
    _assert_argmax("predict flip", pred, ref_sum)


def _against_oracle(m, osd, x, n_classes, scales, flip):
    from dasemanticsegmentationaml_b200 import train as T
    pred = T.predict(m, x, scales=scales, flip=flip)
    assert pred.shape == (x.shape[0],) + tuple(x.shape[2:]) and pred.dtype == torch.uint8
    with torch.no_grad():
        ref, _ = msc_predict(osd, x, n_classes, scales, flip)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            yard, _ = msc_predict(osd, x, n_classes, scales, flip)
    agree = (pred.long() == ref).double().mean().item()
    agree_yard = (yard == ref).double().mean().item()
    print("predict %s scales=%s flip=%s: argmax agreement with fp32 MscEval %.5f, torch-bf16 autocast %.5f"
          % (tuple(x.shape), scales, flip, agree, agree_yard))
    assert agree >= 0.995


@pytest.mark.parametrize("case", [((2, 3, 512, 1024), (0.75, 1.0, 1.25), True),
                                  ((1, 3, 720, 1280), (0.6, 1.0), True),
                                  ((2, 3, 512, 1024), (0.125,), True)],
                         ids=["512x1024-3scales-flip", "720x1280-2scales-flip", "512x1024-smallest-side"])
def test_predict_against_oracle(net19, case):
    m, osd = net19
    shape, scales, flip = case
    x = torch.randn(shape, generator=torch.Generator().manual_seed(5)).to(DEV)
    _against_oracle(m, osd, x, 19, scales, flip)


def test_predict_against_oracle_16_classes(cuda_lib):
    from dasemanticsegmentationaml_b200.model import BiSeNet
    sd = O.make_bisenet_state(seed=0, n_classes=16)
    m = load_oracle_state(BiSeNet("STDCNet813", 16), sd).to(DEV).eval()
    x = torch.randn(2, 3, 512, 1024, generator=torch.Generator().manual_seed(7)).to(DEV)
    _against_oracle(m, to_device(sd, DEV), x, 16, (0.5, 1.0), True)


# ------------------------------------------------------------------ eval_batch / val
class _SameLogits(object):
    """forward_lowres that returns the first result again for an input it has seen.  The forward sums some
    reductions with fp32 atomics, so two forwards of one input can differ in the last bits; with this, two
    evaluations of one batch see the same logits and must agree bit for bit."""

    def __init__(self, fn):
        self.fn, self.seen = fn, []

    def __call__(self, x):
        for k, v in self.seen:
            if k.shape == x.shape and torch.equal(k, x):
                return v
        v = self.fn(x)
        self.seen.append((x.clone(), v))
        return v


def _batches(n_batches, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        labels = torch.randint(0, 20, (2, 256, 512), generator=g)
        labels[labels == 19] = 255
        out.append((torch.randn(2, 3, 256, 512, generator=g).to(DEV), labels.to(DEV)))
    return out


def test_eval_default_path_unchanged(net19):
    from dasemanticsegmentationaml_b200 import losses as L
    from dasemanticsegmentationaml_b200 import train as T
    from dasemanticsegmentationaml_b200.utils import fast_hist_device
    m, _ = net19
    (x, labels), = _batches(1, seed=21)
    m.forward_lowres = _SameLogits(m.forward_lowres)
    try:
        h0, p0 = T.eval_batch(m, x, labels)
        h1, p1 = T.eval_batch(m, x, labels, scales=(1.0,), flip=False)
        with torch.no_grad():   # the single-scale evaluation as it was written before multi-scale support
            p2 = L.upsample_argmax(m.forward_lowres(x)[0], 256, 512, 19, torch.uint8)
            h2 = fast_hist_device(labels.long(), p2, 19, None)
        assert torch.equal(p0, p1) and torch.equal(p0, p2)
        assert torch.equal(h0, h1) and torch.equal(h0, h2)
        r0 = T.val(m, [(x, labels)])
        v0 = T.val.last_hist.clone()
        r1 = T.val(m, [(x, labels)], scales=(1.0,), flip=False)
        assert r0[0] == r1[0] and torch.equal(v0, T.val.last_hist) and torch.equal(v0, h0)
    finally:
        del m.forward_lowres


def test_val_multiscale_sums_batch_histograms(net19):
    from dasemanticsegmentationaml_b200 import train as T
    m, _ = net19
    batches = _batches(3, seed=22)
    scales = (0.75, 1.0, 1.25)
    m.forward_lowres = _SameLogits(m.forward_lowres)
    try:
        T.val(m, batches, scales=scales, flip=True)
        total = T.val.last_hist.clone()
        per = sum(T.eval_batch(m, x, y, scales=scales, flip=True)[0] for x, y in batches)
        assert torch.equal(total, per)
        assert int(total.sum()) > 0
    finally:
        del m.forward_lowres


def test_successive_forwards_do_not_alias(net19):
    """predict keeps every scale's map until the combine: a later forward must not reuse an earlier map's memory."""
    m, _ = net19
    g = torch.Generator().manual_seed(23)
    x1, x2 = torch.randn(2, 3, 256, 512, generator=g).to(DEV), torch.randn(2, 3, 256, 512, generator=g).to(DEV)
    with torch.no_grad():
        a = m.forward_lowres(x1)[0]
        a_copy = a.clone()
        b = m.forward_lowres(x2)[0]
    sa, sb = a.untyped_storage(), b.untyped_storage()
    a0, b0 = sa.data_ptr(), sb.data_ptr()
    assert a0 + sa.nbytes() <= b0 or b0 + sb.nbytes() <= a0
    assert torch.equal(a, a_copy)
