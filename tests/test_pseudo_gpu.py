"""Pseudo-labels for target-domain self-training, from the csrc kernels up to train.predict_confidence /
pseudo_label_thresholds / pseudo_labels.

Kernel level: msc_confidence against msc_argmax (bit-identical class map) and the float64 softmax sum (conf);
the per-class selection bit-exact against a torch restatement (boolean mask, descending sort of the
order-preserving keys, index k_c - 1, min with cap), also over more than 2^32 pixels of one class; the apply
bit-exact against torch.where.  Model level: predict_confidence teacher-forced and against the fp32 MscEval
restatement of tests/test_tta_gpu.py, a whole round (thresholds, labels, supervised_loss) against torch."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import segnet_oracle as O
from tests.helpers import load_oracle_state, to_device
from tests.test_tta_gpu import OUT_HW, _assert_argmax, _maps, _round4, msc_predict

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64 = torch.float64


# ------------------------------------------------------------------ msc_confidence
@pytest.mark.parametrize("ld_kind", ["tight", "32"])
@pytest.mark.parametrize("n_classes", [2, 3, 13, 16, 19, 24, 32])
@pytest.mark.parametrize("n_maps", [1, 2, 5, 12, 16])
def test_msc_confidence_against_float64(cuda_lib, n_maps, n_classes, ld_kind):
    from dasemanticsegmentationaml_b200 import kernels as K
    ld = _round4(n_classes) if ld_kind == "tight" else 32
    n = 1 + n_maps % 3
    views, flags, ref_sum = _maps(n_maps, n_classes, ld, n, seed=1000 * n_maps + n_classes)
    if n_maps == 1:   # one map: also run it mirrored
        flags = [True]
        ref_sum = torch.softmax(torch.flip(F.interpolate(views[0][..., :n_classes].double().permute(0, 3, 1, 2),
                                                         OUT_HW, mode="bilinear", align_corners=True), dims=[3]), dim=1)
    pred = torch.full((n,) + OUT_HW, 255, dtype=torch.uint8, device=DEV)
    conf = torch.full((n,) + OUT_HW, float("nan"), device=DEV)
    K.msc_confidence(views, flags, OUT_HW[0], OUT_HW[1], n_classes, pred, conf)
    argmax = torch.full_like(pred, 255)
    K.msc_argmax(views, flags, OUT_HW[0], OUT_HW[1], n_classes, argmax)
    assert torch.equal(pred, argmax)
    _assert_argmax("msc_confidence %d maps %d classes ld %d" % (n_maps, n_classes, ld), pred, ref_sum)
    want = ref_sum.gather(1, pred.long()[:, None])[:, 0] / n_maps
    err = (conf.double() - want).abs().max().item()
    print("msc_confidence %d maps %d classes: max |conf - float64| %.3g" % (n_maps, n_classes, err))
    assert err <= 1e-5


def test_msc_confidence_refuses_malformed(cuda_lib):
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200._lib import B200Error
    lr = torch.zeros(1, 8, 8, 32, device=DEV)
    pred = torch.empty(1, 32, 32, dtype=torch.uint8, device=DEV)
    conf = torch.empty(1, 32, 32, device=DEV)
    K.msc_confidence([lr] * 16, [False] * 16, 32, 32, 19, pred, conf)
    assert torch.allclose(conf, torch.full_like(conf, 1 / 19))
    with pytest.raises(B200Error, match="maps"):
        K.msc_confidence([lr] * 17, [False] * 17, 32, 32, 19, pred, conf)
    with pytest.raises(B200Error, match="stride"):
        K.msc_confidence([torch.zeros(1, 8, 8, 30, device=DEV)], [True], 32, 32, 19, pred, conf)
    for bad in (1, 33):
        with pytest.raises(B200Error, match="classes"):
            K.msc_confidence([lr], [False], 32, 32, bad, pred, conf)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ per-class selection
def order_key(c):
    """The order-preserving int64 key of fp32 values (csrc/pseudo.cu order_key)."""
    u = c.contiguous().view(torch.int32).long() & 0xFFFFFFFF
    return torch.where(u >= 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000)


def ref_select(preds, confs, n, portion, cap):
    """thr fp32 [n], counts int64 [n]: the definition restated with a boolean mask and a descending sort."""
    p = torch.cat([t.reshape(-1) for t in preds]).long()
    c = torch.cat([t.reshape(-1) for t in confs])
    cap32 = torch.tensor(cap, dtype=torch.float32, device=c.device)
    thr, counts = [], []
    for cl in range(n):
        m = (p == cl) & ~torch.isnan(c)
        cnt = int(m.sum())
        counts.append(cnt)
        if cnt == 0:
            thr.append(cap32)
            continue
        k = min(cnt, max(1, math.ceil(portion * cnt)))
        vals = c[m]
        v = vals[torch.sort(order_key(vals), descending=True, stable=True).indices[k - 1]]
        thr.append(torch.minimum(v, cap32))
    return torch.stack(thr), torch.tensor(counts, dtype=torch.int64, device=c.device)


def _assert_same(got, want):
    thr, counts = got
    rthr, rcounts = want
    assert torch.equal(counts, rcounts), (counts, rcounts)
    assert torch.equal(thr.view(torch.int32), rthr.view(torch.int32)), (thr, rthr)


SHAPES = [(2, 67, 129), (1, 31, 45), (3, 50, 77)]


def _select_data(n, seed, shapes=SHAPES):
    """Batches with ties (50 levels), an all-equal class, an absent class, a one-pixel class, predictions >= n
    (ignored), NaN, negative values and +-0."""
    g = torch.Generator().manual_seed(seed)
    preds, confs = [], []
    for shape in shapes:
        p = torch.randint(0, n + 2, shape, generator=g)
        p[p == n + 1] = 255
        lv = torch.randint(1, 51, shape, generator=g).float() / 50
        c = torch.where(torch.rand(shape, generator=g) < 0.5, lv, torch.rand(shape, generator=g))
        u = torch.rand(shape, generator=g)
        c[u < 0.02] = float("nan")
        c[(u >= 0.02) & (u < 0.04)] = -c[(u >= 0.02) & (u < 0.04)]
        c[(u >= 0.04) & (u < 0.05)] = 0.0
        c[(u >= 0.05) & (u < 0.06)] = -0.0
        c[p == 1] = 0.75                     # all-equal class
        if n > 2:
            p[p == 2] = 0                    # absent class
        preds.append(p.to(torch.uint8))
        confs.append(c.float())
    if n > 3:                                # class 3: one pixel in the whole set
        for p in preds:
            p[p == 3] = 0
        preds[0].view(-1)[5] = 3
        confs[0].view(-1)[5] = 0.3
    return [p.to(DEV) for p in preds], [c.to(DEV) for c in confs]


@pytest.mark.parametrize("portion", [1e-9, 0.2, 0.5, 1.0])
@pytest.mark.parametrize("n", [2, 19, 32])
def test_thresholds_bit_exact(cuda_lib, n, portion):
    from dasemanticsegmentationaml_b200 import train as T
    preds, confs = _select_data(n, seed=100 * n + int(portion * 10))
    for cap in (0.9, 1.0):
        want = ref_select(preds, confs, n, portion, cap)
        got = T.pseudo_label_thresholds(preds, confs, n, portion, cap)
        _assert_same(got, want)
        if n > 3:
            assert int(got[1][2]) == 0 and float(got[0][2]) == torch.tensor(cap).item()
            assert int(got[1][3]) == 1
    # the same pixels as one batch, and split into batches of other sizes (offset views: the scalar path)
    flat_p = torch.cat([p.reshape(-1) for p in preds])
    flat_c = torch.cat([c.reshape(-1) for c in confs])
    want = ref_select(preds, confs, n, portion, 0.9)
    _assert_same(T.pseudo_label_thresholds([flat_p], [flat_c], n, portion, 0.9), want)
    cuts = [0, 1, 1000, 1013, 9000, flat_p.numel()]
    _assert_same(T.pseudo_label_thresholds([flat_p[a:b] for a, b in zip(cuts, cuts[1:])],
                                           [flat_c[a:b] for a, b in zip(cuts, cuts[1:])], n, portion, 0.9), want)


def test_select_kernels_direct(cuda_lib):
    """The four hist / pick rounds through the kernels' wrappers, reused for a second selection (the picks
    leave hist zero), and their refusals."""
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200._lib import B200Error
    n = 19
    preds, confs = _select_data(n, seed=7)
    state = torch.empty(3 * n, dtype=torch.int64, device=DEV)
    hist = torch.zeros(n * 256, dtype=torch.int64, device=DEV)
    thr = torch.empty(n, device=DEV)
    counts = torch.empty(n, dtype=torch.int64, device=DEV)
    for portion in (0.5, 0.3):
        for pass_ in range(4):
            for p, c in zip(preds, confs):
                K.class_select_hist(p, c, n, pass_, state, hist)
            K.class_select_pick(n, pass_, portion, 0.9, state, hist, thr, counts)
        _assert_same((thr, counts), ref_select(preds, confs, n, portion, 0.9))
        assert int(hist.abs().sum()) == 0
    p, c = preds[0], confs[0]
    with pytest.raises(B200Error, match="pass"):
        K.class_select_hist(p, c, n, 4, state, hist)
    with pytest.raises(B200Error, match="classes"):
        K.class_select_hist(p, c, 33, 0, state, hist)
    for bad in (0.0, 1.5, float("nan")):
        with pytest.raises(B200Error, match="portion"):
            K.class_select_pick(n, 0, bad, 0.9, state, hist, thr, counts)
        with pytest.raises(B200Error, match="cap"):
            K.class_select_pick(n, 0, 0.5, bad, state, hist, thr, counts)
    with pytest.raises(B200Error, match="pass"):
        K.class_select_pick(n, -1, 0.5, 0.9, state, hist, thr, counts)
    torch.cuda.synchronize()


def test_counts_above_2_to_32(cuda_lib):
    """Five copies of one 2^30-pixel batch: class 0 holds ~4.8 G pixels.  conf takes 1000 levels, so the
    expected k-th value follows exactly from a bincount of the levels."""
    from dasemanticsegmentationaml_b200 import train as T
    g = torch.Generator(device=DEV).manual_seed(3)
    npx = 1 << 30
    levels = torch.linspace(0.05, 1.0, 1000, device=DEV)
    idx = torch.randint(0, 1000, (npx,), device=DEV, generator=g, dtype=torch.int16)
    pred = (torch.rand(npx, device=DEV, generator=g) < 0.1).to(torch.uint8)
    conf = levels[idx.long()]
    per = torch.bincount(pred.long() * 1000 + idx.long(), minlength=2000).view(2, 1000).cpu() * 5
    del idx
    torch.cuda.empty_cache()
    for portion in (0.5, 0.2):
        thr, counts = T.pseudo_label_thresholds([pred] * 5, [conf] * 5, 2, portion, 0.9)
        for c in range(2):
            cnt = int(per[c].sum())
            k = min(cnt, max(1, math.ceil(portion * cnt)))
            from_top = torch.flip(per[c], dims=[0]).cumsum(0)
            lv = 999 - int(torch.searchsorted(from_top, torch.tensor(k)))
            want = min(levels[lv].item(), torch.tensor(0.9).item())
            assert int(counts[c]) == cnt
            assert float(thr[c]) == want, (c, portion, float(thr[c]), want)
        assert int(counts[0]) > 1 << 32


# ------------------------------------------------------------------ apply
@pytest.mark.parametrize("n", [2, 19, 32])
def test_apply_bit_exact(cuda_lib, n):
    from dasemanticsegmentationaml_b200 import kernels as K
    from dasemanticsegmentationaml_b200 import train as T
    preds, confs = _select_data(n, seed=n)
    thr = torch.rand(n, generator=torch.Generator().manual_seed(n)).to(DEV)
    for p, c in zip(preds, confs):
        pl = p.long()
        keep = (pl < n) & (c >= thr[pl.clamp(max=n - 1)])
        want = torch.where(keep, pl, torch.full_like(pl, 255))
        assert torch.equal(T.pseudo_labels(p, c, thr), want)
        assert torch.equal(T.pseudo_labels(p, c, thr, dtype=torch.uint8), want.to(torch.uint8))
        inplace = p.clone()
        K.pseudo_label_apply(inplace, c, n, thr, inplace)
        assert torch.equal(inplace, want.to(torch.uint8))
        glob = torch.where(c >= 0.6, pl, torch.full_like(pl, 255))    # one global threshold
        assert torch.equal(T.pseudo_labels(p, c, 0.6), torch.where(pl < 32, glob, torch.full_like(pl, 255)))


# ------------------------------------------------------------------ the network
@pytest.fixture(scope="module")
def net19(cuda_lib):
    from dasemanticsegmentationaml_b200.model import BiSeNet
    sd = O.make_bisenet_state(seed=0)
    return load_oracle_state(BiSeNet("STDCNet813", 19), sd).to(DEV).eval(), to_device(sd, DEV)


class _Recorder(object):
    """forward_lowres that keeps every result (to restate the combine over the model's own maps)."""

    def __init__(self, fn):
        self.fn, self.out = fn, []

    def __call__(self, x):
        v = self.fn(x)
        self.out.append(v)
        return v


def test_predict_confidence_teacher_forced(net19):
    from dasemanticsegmentationaml_b200 import losses as L
    from dasemanticsegmentationaml_b200 import train as T
    m, osd = net19
    x = torch.randn(2, 3, 256, 512, generator=torch.Generator().manual_seed(31)).to(DEV)
    scales = (0.75, 1.0, 1.25)
    m.forward_lowres = _Recorder(m.forward_lowres)
    try:
        pred, conf = T.predict_confidence(m, x, scales=scales, flip=True)
        runs = m.forward_lowres.out
    finally:
        del m.forward_lowres
    assert pred.shape == conf.shape == (2, 256, 512) and pred.dtype == torch.uint8 and conf.dtype == torch.float32
    assert len(runs) == 3
    ref_sum = 0
    maps, flags = [], []
    for r in runs:
        lr = r[0]
        for half, mirrored in ((lr[:2], False), (lr[2:], True)):
            up = F.interpolate(half[..., :19].double().permute(0, 3, 1, 2), (256, 512), mode="bilinear",
                               align_corners=True)
            p = torch.softmax(up, dim=1)
            ref_sum = ref_sum + (torch.flip(p, dims=[3]) if mirrored else p)
            maps.append(half)
            flags.append(mirrored)
    _assert_argmax("predict_confidence flip", pred, ref_sum)
    err = (conf.double() - ref_sum.gather(1, pred.long()[:, None])[:, 0] / 6).abs().max().item()
    print("predict_confidence: max |conf - float64| %.3g" % err)
    assert err <= 1e-5
    # predict's combine over the same maps gives the same class map
    assert torch.equal(L.multiscale_argmax(maps, flags, 256, 512, 19, torch.uint8), pred)
    # and the class map agrees with the fp32 MscEval restatement over the oracle
    with torch.no_grad():
        ref, _ = msc_predict(osd, x, 19, scales, True)
    agree = (pred.long() == ref).double().mean().item()
    print("predict_confidence vs fp32 MscEval: argmax agreement %.5f" % agree)
    assert agree >= 0.995


def test_predict_confidence_single_scale(net19):
    """One scale, no flip: one map, the softmax of the up-sampled logits at the argmax."""
    from dasemanticsegmentationaml_b200 import train as T
    m, _ = net19
    x = torch.randn(2, 3, 128, 256, generator=torch.Generator().manual_seed(32)).to(DEV)
    m.forward_lowres = _Recorder(m.forward_lowres)
    try:
        pred, conf = T.predict_confidence(m, x)
        (lr,) = [r[0] for r in m.forward_lowres.out]
    finally:
        del m.forward_lowres
    up = F.interpolate(lr[..., :19].double().permute(0, 3, 1, 2), (128, 256), mode="bilinear", align_corners=True)
    p = torch.softmax(up, dim=1)
    _assert_argmax("predict_confidence single", pred, p)
    assert (conf.double() - p.gather(1, pred.long()[:, None])[:, 0]).abs().max().item() <= 1e-5


def test_pseudo_label_round(net19):
    """predict_confidence over three batches -> thresholds -> labels -> supervised_loss, each against torch."""
    from dasemanticsegmentationaml_b200 import train as T
    m, _ = net19
    g = torch.Generator().manual_seed(33)
    xs = [torch.randn(2, 3, 256, 512, generator=g).to(DEV) for _ in range(3)]
    preds, confs = zip(*[T.predict_confidence(m, x, scales=(1.0,), flip=True) for x in xs])
    thr, counts = T.pseudo_label_thresholds(preds, confs, 19, 0.5, 0.9)
    want = ref_select(preds, confs, 19, 0.5, 0.9)
    _assert_same((thr, counts), want)
    assert int(counts.sum()) == 3 * 2 * 256 * 512
    for x, p, c in zip(xs, preds, confs):
        labels = T.pseudo_labels(p, c, thr)
        pl = p.long()
        assert torch.equal(labels, torch.where(c >= want[0][pl], pl, torch.full_like(pl, 255)))
        assert 0 < int((labels == 255).sum()) < labels.numel()
        loss, lr = T.supervised_loss(m, x, labels)
        ref = sum(F.cross_entropy(F.interpolate(t[..., :19].float().permute(0, 3, 1, 2), (256, 512), mode="bilinear",
                                                align_corners=True), labels, ignore_index=255) for t in lr)
        print("supervised_loss on pseudo-labels %.6f, torch %.6f" % (loss.item(), ref.item()))
        assert abs(loss.item() - ref.item()) < 1e-4 * abs(ref.item())
