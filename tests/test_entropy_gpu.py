"""ADVENT (Vu et al., CVPR 2019) on the fused up-sampling: csrc/entropy.cu's kernels against float64 torch, the
autograd nodes of losses.upsample_entropy / upsample_self_information, and train.train_minent_step /
train_advent_step against an fp32 restatement of ADVENT's MinEnt / AdvEnt iterations over the oracle network.

The ADVENT formulas are restated here (the oracle package is left as it is):
  prob_2_entropy(p) = -p * log2(p + 1e-30) / log2(C)
  entropy_loss(p)   = -sum(p * log2(p + 1e-30)) / (N * H * W * log2(C))
applied to softmax(F.interpolate(logits, bilinear, align_corners=True))."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import segnet_oracle as O
from tests.helpers import assert_within, bf16_ulp, cosine, gate, load_oracle_state, rel_l2, to_device
from tests.test_classes_gpu import _disc_cls, _seg

pytestmark = pytest.mark.gpu
DEV = "cuda"
F64 = torch.float64
COUNTS = [2, 13, 16, 19, 32]
# (h_lr, w_lr, H, W): factor 8, factor 16 and the non-integer factors of 720 x 1280
SHAPES = {"x8": (16, 32, 128, 256), "x16": (8, 16, 128, 256), "720_from_90": (90, 160, 720, 1280),
          "720_from_45": (45, 80, 720, 1280)}


def prob_2_entropy(p):
    c = p.shape[1]
    return -torch.mul(p, torch.log2(p + 1e-30)) / math.log2(c)


def entropy_loss(p):
    n, c, h, w = p.shape
    return -torch.sum(torch.mul(p, torch.log2(p + 1e-30))) / (n * h * w * math.log2(c))


def _logits(n_classes, shape, ld, seed):
    """fp32 [2, h, w, ld] with NaN padding floats: image 0 at 3*randn, image 1 spread uniformly over +-80 (most
    fp32 probabilities underflow to 0 there)."""
    h, w, H, W = SHAPES[shape]
    g = torch.Generator().manual_seed(seed)
    lr = torch.full((2, h, w, ld), float("nan"))
    lr[0, ..., :n_classes] = 3 * torch.randn(h, w, n_classes, generator=g)
    lr[1, ..., :n_classes] = 160 * torch.rand(h, w, n_classes, generator=g) - 80
    return lr.to(DEV), H, W


def _ref_leaf(lr, n_classes):
    return lr[..., :n_classes].double().clone().requires_grad_(True)


def _axis(n_in, n_out):
    """F.interpolate's fp32 align_corners=True source indices and weights (the kernels use the same arithmetic)."""
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    src = np.arange(n_out, dtype=np.float32) * scale
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = i0 + (i0 < n_in - 1)
    l1 = src - i0.astype(np.float32)
    l0 = np.float32(1) - l1
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dt)  # noqa: E731
    return t(i0, torch.int64), t(i1, torch.int64), t(l0, F64), t(l1, F64)


def _probs64(leaf, H, W):
    """float64 bilinear up-sampling of the float64 leaf [N, h, w, n] with fp32 F.interpolate's indices and
    weights -> (z [N, n, H, W], softmax(z))."""
    _, h, w, _ = leaf.shape
    i0, i1, a0, a1 = _axis(h, H)
    j0, j1, b0, b1 = _axis(w, W)
    rows = leaf[:, i0] * a0[None, :, None, None] + leaf[:, i1] * a1[None, :, None, None]
    z = (rows[:, :, j0] * b0[None, None, :, None] + rows[:, :, j1] * b1[None, None, :, None]).permute(0, 3, 1, 2)
    return z, torch.softmax(z, dim=1)


def test_reference_interpolation_is_f_interpolate(cuda_lib):
    g = torch.Generator().manual_seed(2)
    for h, w, H, W in SHAPES.values():
        leaf = (3 * torch.randn(2, h, w, 5, generator=g)).to(DEV, F64)
        z, _ = _probs64(leaf, H, W)
        ref = F.interpolate(leaf.permute(0, 3, 1, 2), (H, W), mode="bilinear", align_corners=True)
        # fp32 source positions are off by <= half an ulp of max(h, w) per axis, against corner differences <= 2 max|lr|
        assert (z - ref).abs().max().item() < 4 * 2.0 ** -24 * max(h, w) * leaf.abs().max().item()


def _abs_terms(leaf, z, gz):
    """sum over the output pixels of |interpolation weight * per-pixel gradient| for every low-resolution value."""
    (t,) = torch.autograd.grad(z, leaf, gz.abs(), retain_graph=True)
    return t


def _d_lr_ok(name, got, base, want, terms, n_classes):
    """got = base + the kernel's gradient; padding classes untouched (still base's), the rest within
    1e-5 * sum|terms| + 1e-6 of the float64 gradient."""
    assert torch.isfinite(got[..., :n_classes]).all(), name
    if got.shape[-1] > n_classes:
        assert torch.equal(got[..., n_classes:], base[..., n_classes:]), name
    assert_within(name, got[..., :n_classes].double() - base[..., :n_classes].double(), want,
                  1e-5 * terms + 1e-6)


@pytest.mark.parametrize("ld_kind", ["tight", "32"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("n_classes", COUNTS)
def test_entropy_kernels_against_float64(cuda_lib, n_classes, shape, ld_kind):
    from dasemanticsegmentationaml_b200 import kernels as K
    ld = (n_classes + 3) // 4 * 4 if ld_kind == "tight" else 32
    lr, H, W = _logits(n_classes, shape, ld, seed=n_classes * 7 + len(shape))
    N = lr.shape[0]
    leaf = _ref_leaf(lr, n_classes)
    z, p = _probs64(leaf, H, W)
    I_ref = prob_2_entropy(p)
    S_ref = I_ref.sum()
    E_ref = entropy_loss(p)
    assert abs(S_ref.item() / (N * H * W) - E_ref.item()) <= 1e-12 * abs(E_ref.item())

    # forward, sum only: E, and the accumulator accumulates
    acc = torch.zeros(1, dtype=F64, device=DEV)
    K.entropy_fwd(lr, H, W, n_classes, K.ENT_SUM, acc=acc)
    e1 = acc.item() / (N * H * W)
    K.entropy_fwd(lr, H, W, n_classes, K.ENT_SUM, acc=acc)
    print("n=%d %s ld=%d E %.9f ref %.9f" % (n_classes, shape, ld, e1, E_ref.item()))
    assert abs(e1 - E_ref.item()) <= 1e-5 * abs(E_ref.item())
    assert abs(acc.item() - 2 * e1 * N * H * W) <= 1e-9 * abs(acc.item())

    # forward with the map, both layouts
    maps = {}
    for layout in (K.MAP_PLAIN, K.MAP_ZERO_BORDERED):
        hw = (H, W) if layout == K.MAP_PLAIN else (H + 2, W + 2)
        m = torch.full((N,) + hw + (32,), float("nan"), dtype=torch.bfloat16, device=DEV)
        acc_m = torch.full((1,), 0.25, dtype=F64, device=DEV)
        K.entropy_fwd(lr, H, W, n_classes, K.ENT_MAP, emap=m, layout=layout, acc=acc_m)
        assert abs((acc_m.item() - 0.25) / (N * H * W) - E_ref.item()) <= 1e-5 * abs(E_ref.item())
        inner = m if layout == K.MAP_PLAIN else m[:, 1:H + 1, 1:W + 1]
        if layout == K.MAP_ZERO_BORDERED:
            border = torch.cat([m[:, 0].flatten(), m[:, -1].flatten(), m[:, :, 0].flatten(), m[:, :, -1].flatten()])
            assert torch.equal(border.float(), torch.zeros_like(border.float())), "border not zero"
        assert torch.equal(inner[..., n_classes:].float(), torch.zeros_like(inner[..., n_classes:].float()))
        got = inner[..., :n_classes].permute(0, 3, 1, 2).double()
        assert torch.isfinite(got).all()
        want = I_ref.detach()
        assert_within("I map n=%d %s layout %d" % (n_classes, shape, layout), got, want, bf16_ulp(want) + 1e-6)
        maps[layout] = inner.clone()
    assert torch.equal(maps[K.MAP_PLAIN], maps[K.MAP_ZERO_BORDERED])
    # the map mode also runs without an accumulator
    m = torch.empty((N, H, W, 32), dtype=torch.bfloat16, device=DEV)
    K.entropy_fwd(lr, H, W, n_classes, K.ENT_MAP, emap=m)
    assert torch.equal(m, maps[K.MAP_PLAIN])

    # backward mode 0: the entropy training pass (sum and unscaled gradient, one pass), accumulating
    (gz,) = torch.autograd.grad(S_ref, z, retain_graph=True)
    (g_ref,) = torch.autograd.grad(S_ref, leaf, retain_graph=True)
    terms = _abs_terms(leaf, z, gz)
    base = torch.randn(lr.shape, generator=torch.Generator().manual_seed(3)).to(DEV)
    d_lr = base.clone()
    acc_t = torch.full((1,), 1.5, dtype=F64, device=DEV)
    K.entropy_bwd(lr, H, W, n_classes, K.ENT_TRAIN, d_lr, acc=acc_t)
    assert abs((acc_t.item() - 1.5) / (N * H * W) - E_ref.item()) <= 1e-5 * abs(E_ref.item())
    _d_lr_ok("entropy grad n=%d %s ld=%d" % (n_classes, shape, ld), d_lr, base, g_ref, terms, n_classes)

    # backward mode 1: self-information backward from a bf16 dI, plain and zero-bordered, accumulating
    g = torch.Generator().manual_seed(5)
    dI = (torch.randn(N, H, W, 32, generator=g) * 0.01).to(torch.bfloat16)
    dI[..., n_classes:] = float("nan")                      # padding channels are never read
    dI = dI.to(DEV)
    dI64 = dI[..., :n_classes].permute(0, 3, 1, 2).double()
    (gz1,) = torch.autograd.grad((I_ref * dI64).sum(), z, retain_graph=True)
    (g1_ref,) = torch.autograd.grad((I_ref * dI64).sum(), leaf, retain_graph=True)
    terms1 = _abs_terms(leaf, z, gz1)
    bordered = torch.full((N, H + 2, W + 2, 32), float("nan"), dtype=torch.bfloat16, device=DEV)
    bordered[:, 1:H + 1, 1:W + 1] = dI
    for layout, dmap in ((K.MAP_PLAIN, dI), (K.MAP_ZERO_BORDERED, bordered)):
        d_lr = base.clone()
        K.entropy_bwd(lr, H, W, n_classes, K.ENT_SELF_INFO, d_lr, d_map=dmap, layout=layout)
        _d_lr_ok("self-info grad n=%d %s ld=%d layout %d" % (n_classes, shape, ld, layout), d_lr, base, g1_ref,
                 terms1, n_classes)


def test_upsample_entropy_autograd(cuda_lib):
    from dasemanticsegmentationaml_b200 import losses as L
    n_classes = 19
    lr, H, W = _logits(n_classes, "x8", 32, seed=1)
    lr = torch.nan_to_num(lr, nan=0.0)
    with torch.no_grad():
        e_ng = L.upsample_entropy(lr, H, W, n_classes)
    a = lr.clone().requires_grad_(True)
    e = L.upsample_entropy(a, H, W, n_classes)
    assert e.dtype == torch.float32 and e.dim() == 0
    print("entropy with grad %.9f without %.9f" % (e.item(), e_ng.item()))
    assert abs(e.item() - e_ng.item()) <= 1e-6 * abs(e_ng.item())
    (3.0 * e).backward()
    leaf = _ref_leaf(lr, n_classes)
    z, p = _probs64(leaf, H, W)
    E = entropy_loss(p)
    assert abs(e.item() - E.item()) <= 1e-5 * abs(E.item())
    (gz,) = torch.autograd.grad(3.0 * E, z, retain_graph=True)
    (g_ref,) = torch.autograd.grad(3.0 * E, leaf, retain_graph=True)
    terms = _abs_terms(leaf, z, gz)
    assert float(a.grad[..., n_classes:].abs().max()) == 0.0
    assert_within("upsample_entropy grad", a.grad[..., :n_classes].double(), g_ref,
                  1e-5 * terms + 3e-6 / (lr.shape[0] * H * W))


@pytest.mark.parametrize("shape", [(2, 16, 32, 128, 256), (1, 12, 20, 96, 160)])
def test_self_information_feeds_the_dense_discriminator_pair_view(cuda_lib, shape):
    """upsample_self_information(zero_border=True) through FCDiscriminator's pair view against the same module on
    the plain layout, with the gates of test_modules_gpu.py::test_dense_discriminator_pair_view."""
    from dasemanticsegmentationaml_b200 import losses as L
    from dasemanticsegmentationaml_b200.model import FCDiscriminator
    from dasemanticsegmentationaml_b200.model._glue import ZeroBordered, zero_bordered_base
    n, h, w, H, W = shape
    d = load_oracle_state(FCDiscriminator(19), O.make_discriminator_state("dense", seed=11)).to(DEV).train()
    g = torch.Generator().manual_seed(21)
    lr = torch.zeros(n, h, w, 32)
    lr[..., :19] = 3 * torch.randn(n, h, w, 19, generator=g)
    lr = lr.to(DEV)
    res = []
    for zb in (False, True):
        a = lr.clone().requires_grad_(True)
        m = L.upsample_self_information(a, H, W, zero_border=zb)
        assert m.shape == (n, 19, H, W) and m.dtype == torch.bfloat16
        if zb:
            assert isinstance(m, ZeroBordered)
            base = zero_bordered_base(m)
            assert base is not None and base.shape == (n, H + 2, W + 2, 32)
            assert zero_bordered_base(m.detach()) is not None
            border = torch.cat([base[:, 0].flatten(), base[:, -1].flatten(), base[:, :, 0].flatten(), base[:, :, -1].flatten()])
            assert float(border.float().abs().max()) == 0.0
            assert float(base[..., 19:].float().abs().max()) == 0.0
            assert torch.equal(m, res[0][4])
        else:
            assert not isinstance(m, ZeroBordered)
        d.zero_grad()
        y = d(m)
        loss = L.bce_with_logits_const(y, 0.0)
        loss.backward()
        assert torch.isfinite(a.grad).all()
        res.append((y.detach().clone(), a.grad.clone(), {k: v.grad.clone() for k, v in d.named_parameters()},
                    loss.item(), m.detach().clone()))
    (y0, g0, pg0, l0, _), (y1, g1, pg1, l1, _) = res
    print("self-information pair view: out", rel_l2(y1, y0), "d_lr", rel_l2(g1, g0), "loss", l0, l1)
    assert rel_l2(y1, y0) < 5e-3
    assert abs(l1 - l0) < 1e-3 * abs(l0)
    for k in pg0:
        gate("self-info pair view %s" % k, cosine(pg1[k], pg0[k]), 0.9995)
        assert rel_l2(pg1[k], pg0[k]) < 3e-2, k
    gate("self-info pair view d_lr", cosine(g1, g0), 0.9995)
    assert rel_l2(g1, g0) < 3e-2


def test_self_information_odd_size_is_a_plain_view(cuda_lib):
    from dasemanticsegmentationaml_b200 import losses as L
    from dasemanticsegmentationaml_b200.model._glue import ZeroBordered
    lr = torch.randn(1, 13, 17, 32, device=DEV)
    m = L.upsample_self_information(lr, 97, 129, 19, zero_border=True)
    assert not isinstance(m, ZeroBordered) and m.shape == (1, 19, 97, 129)


# ----------------------------------------------------------------------------- the two steps
def _o_minent(seg_sd, images, labels, images_t, opt, lambda_ent):
    """ADVENT's MinEnt iteration on this project's supervised loss, fp32."""
    opt.zero_grad()
    loss, _ = O.supervised_loss(seg_sd, images, labels, True)
    loss.backward()
    out_t = O.bisenet_forward(seg_sd, images_t, True)[0]
    loss_ent = entropy_loss(F.softmax(out_t, dim=1))
    (lambda_ent * loss_ent).backward()
    opt.step()
    return float(loss), float(loss_ent)


def _o_advent(seg_sd, d_sd, kind, images, labels, images_t, opt, opt_d, lambda_adv):
    """ADVENT's train_advent iteration on this project's supervised loss, fp32: accumulated gradients, one step
    per optimizer, halved discriminator losses."""
    d_params = [v for v in d_sd.values() if v.is_floating_point() and v.requires_grad]
    opt.zero_grad()
    opt_d.zero_grad()
    for p in d_params:
        p.requires_grad_(False)
    loss, (out, _, _) = O.supervised_loss(seg_sd, images, labels, True)
    loss.backward()
    out_t = O.bisenet_forward(seg_sd, images_t, True)[0]
    d_out = O.discriminator_forward(kind, d_sd, prob_2_entropy(F.softmax(out_t, dim=1)))
    loss_adv = O.bce_with_logits_const(d_out, 0.0)
    (lambda_adv * loss_adv).backward()
    for p in d_params:
        p.requires_grad_(True)
    out, out_t = out.detach(), out_t.detach()
    loss_d_src = O.bce_with_logits_const(O.discriminator_forward(kind, d_sd, prob_2_entropy(F.softmax(out, dim=1))), 0.0) / 2
    loss_d_src.backward()
    loss_d_tgt = O.bce_with_logits_const(O.discriminator_forward(kind, d_sd, prob_2_entropy(F.softmax(out_t, dim=1))), 1.0) / 2
    loss_d_tgt.backward()
    opt.step()
    opt_d.step()
    return float(loss), float(loss_adv), float(loss_d_src), float(loss_d_tgt)


def _inputs(n_classes, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(2, 3, 128, 256, generator=g).to(DEV)
    xt = torch.randn(2, 3, 128, 256, generator=g).to(DEV)
    labels = torch.randint(0, n_classes, (2, 128, 256), generator=g).to(DEV)
    return x, labels, xt


def _check_losses(got, want):
    print("step losses", got, want)
    assert all(np.isfinite(got))
    assert abs(got[0] - want[0]) / want[0] < 3e-2
    for a, b in zip(got[1:], want[1:]):
        assert abs(a - b) < 0.1 * max(1.0, abs(b))


KEY = "conv_out.conv_out.weight"


def test_minent_step_matches_restatement(cuda_lib):
    from dasemanticsegmentationaml_b200 import train as T
    n_classes = 19
    m, sd = _seg(n_classes, seed=21)
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    x, labels, xt = _inputs(n_classes, 10)
    w0 = m.state_dict()[KEY].clone()
    got = [float(v) for v in T.train_minent_step(m, opt, x, labels, xt, lambda_ent=0.01)]
    osd = to_device(sd, DEV, True)
    o_opt = torch.optim.SGD([v for v in osd.values() if v.requires_grad], lr=0.01, momentum=0.9, weight_decay=5e-4)
    o0 = osd[KEY].detach().clone()
    want = _o_minent(osd, x, labels, xt, o_opt, 0.01)
    _check_losses(got, want)
    c = cosine(m.state_dict()[KEY] - w0, osd[KEY].detach() - o0)
    print("minent step: update cosine of", KEY, c)
    assert c > 0.9


@pytest.mark.parametrize("n_classes, kind", [(19, "dense"), (19, "dwsep_bn"), (19, "dwsep"), (16, "dense"),
                                             (16, "dwsep_bn")])
def test_advent_step_matches_restatement(cuda_lib, n_classes, kind):
    from dasemanticsegmentationaml_b200 import train as T
    m, sd = _seg(n_classes, seed=21)
    dsd = O.make_discriminator_state(kind, seed=4, n_classes=n_classes)
    d = load_oracle_state(_disc_cls(kind)(n_classes), dsd).to(DEV)
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    opt_d = torch.optim.Adam(d.parameters(), lr=1e-3, betas=(0.9, 0.99))
    x, labels, xt = _inputs(n_classes, 10)
    w0 = m.state_dict()[KEY].clone()
    got = [float(v) for v in T.train_advent_step(m, d, opt, opt_d, x, labels, xt, lambda_adv=0.01)]
    osd, odsd = to_device(sd, DEV, True), to_device(dsd, DEV, True)
    o_opt = torch.optim.SGD([v for v in osd.values() if v.requires_grad], lr=0.01, momentum=0.9, weight_decay=5e-4)
    o_opt_d = torch.optim.Adam([v for v in odsd.values() if v.requires_grad], lr=1e-3, betas=(0.9, 0.99))
    o0 = osd[KEY].detach().clone()
    want = _o_advent(osd, odsd, kind, x, labels, xt, o_opt, o_opt_d, 0.01)
    _check_losses(got, want)
    c = cosine(m.state_dict()[KEY] - w0, osd[KEY].detach() - o0)
    print("advent step n=%d %s: update cosine of %s %.5f" % (n_classes, kind, KEY, c))
    assert c > 0.9
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in d.parameters())


@pytest.mark.parametrize("step", ["minent", "advent"])
def test_graphed_steps_match_eager(cuda_lib, step):
    """The CUDA-graph replay of either step trains like the eager launches (gates of
    test_classes_gpu.py::test_graphed_da_step_matches_eager)."""
    from dasemanticsegmentationaml_b200 import optim as B200Optim
    from dasemanticsegmentationaml_b200 import train as T
    from dasemanticsegmentationaml_b200.model import FCDiscriminator
    n_classes = 16
    x, labels, xt = _inputs(n_classes, 12)
    runs = []
    for graphed in (False, True):
        m, _ = _seg(n_classes, seed=21)
        d = load_oracle_state(FCDiscriminator(n_classes), O.make_discriminator_state("dense", seed=4, n_classes=n_classes)).to(DEV)
        opt = B200Optim.FusedSGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
        opt_d = B200Optim.FusedAdam(d.parameters(), lr=1e-3, betas=(0.9, 0.99))

        if step == "minent":
            def fn(images, labels, images_t):
                return T.train_minent_step(m, opt, images, labels, images_t)
        else:
            def fn(images, labels, images_t):
                return T.train_advent_step(m, d, opt, opt_d, images, labels, images_t)

        losses = []
        if graphed:
            gs = T.GraphedStep(fn, dict(images=x, labels=labels, images_t=xt), warmup=1)
            for _ in range(4):
                losses.append([float(v) for v in gs()])
        else:
            fn(x, labels, xt)
            for _ in range(4):
                losses.append([float(v) for v in fn(x, labels, xt)])
        runs.append(losses)
    print(step, "eager  ", runs[0])
    print(step, "graphed", runs[1])
    for u, v in zip(runs[0][0], runs[1][0]):
        assert abs(u - v) < 5e-2 * max(1.0, abs(u)), (runs[0], runs[1])
    for a, b in zip(runs[0], runs[1]):
        assert all(np.isfinite(b))
        assert abs(a[0] - b[0]) < 6e-2 * abs(a[0]), (runs[0], runs[1])
    assert runs[1][3][0] != runs[1][0][0]
