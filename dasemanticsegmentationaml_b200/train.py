"""Training / evaluation steps with the loss composition of the reference's ``train.py``.

``train_step`` is the body of ``train()`` (train.py:76-93), ``train_da_step`` the body of
``train_DA()``'s inner loop (train.py:192-262) and ``val`` the evaluation loop (train.py:24-61),
restated over the fused B200 ops:

* the three cross-entropy terms consume the low-resolution logits directly (bilinear up-sampling,
  log-softmax and NLL fused, nothing of size N x 19 x H x W is written);
* ``softmax(output)`` feeding the discriminator is one fused up-sample+softmax kernel writing bf16;
* BCE-with-logits against all-zeros / all-ones needs no target tensor;
* bf16 needs no loss scaling, so the reference's fp16 ``GradScaler`` (train.py:137,219-221) is gone;
* multi-GPU is one process per GPU: gradients are averaged with one NCCL all-reduce per optimizer
  step (the reference's nn.DataParallel reduce-add, train.py:145-152,497), the evaluation
  confusion matrices are summed with an int64 all-reduce.
"""
import math

import numpy as np
import torch
import torch.distributed as dist

from . import kernels as K
from . import losses
from .utils import compute_global_accuracy, fast_hist_device, per_class_iu


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def allreduce_grads(params, world=None):
    """Average ``.grad`` over ranks with ONE all-reduce over a flat fp32 bucket; parameters whose
    grad is None on this step (dead classifier head, aux heads in the adversarial pass) are skipped
    on every rank alike."""
    world = world or _world()
    if world == 1:
        return
    grads = [p.grad for p in params if p.grad is not None]
    if grads and grads[0].is_cuda:
        # most gradients were already averaged in place, overlapped with the backward (ops.REDUCER)
        from . import ops
        grads = ops.REDUCER.finish(grads)
    if not grads:
        return
    flat = torch._utils._flatten_dense_tensors(grads)
    if dist.get_backend() == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG)
    else:
        dist.all_reduce(flat)
        flat.div_(world)
    torch._foreach_copy_(grads, list(torch._utils._unflatten_dense_tensors(flat, grads)))


def supervised_loss(model, images, labels, loss="ce", ohem_threshold=0.3567, ohem_keep=None):
    """loss1 + loss2 + loss3 over (out, out16, out32)  (train.py:84-89 / 212-217), over the model's
    ``n_classes`` classes."""
    lr = model.forward_lowres(images)
    ncls = model.n_classes
    if loss == "ohem":
        if ohem_keep is None:
            ohem_keep = labels.numel() // 16
        terms = [losses.upsample_ohem_cross_entropy(t, labels, ohem_threshold, ohem_keep, n_classes=ncls) for t in lr]
    else:
        terms = [losses.upsample_cross_entropy(t, labels, n_classes=ncls) for t in lr]
    return terms[0] + terms[1] + terms[2], lr


def train_step(model, optimizer, images, labels, loss="ce", **kw):
    """One supervised iteration (train.py:76-93). Returns the loss tensor (no host sync)."""
    model.train()
    optimizer.zero_grad()
    total, _ = supervised_loss(model, images, labels, loss, **kw)
    total.backward()
    allreduce_grads(_opt_params(optimizer))
    optimizer.step()
    return total.detach()


def _opt_params(optimizer):
    return [p for g in optimizer.param_groups for p in g["params"]]


def _zb(model_D):
    """The dense FCDiscriminator reads its input as 128-byte column pairs of a zero-bordered buffer
    (losses.upsample_softmax(zero_border=True)); the depthwise-separable variants take the plain layout."""
    return bool(getattr(model_D, "wants_zero_bordered_input", False))


def train_da_step(model, model_D, optimizer, optimizer_D, images, labels, images_t, lambda_adv=0.001):
    """One adversarial domain-adaptation iteration (train.py:192-262).

    Returns (loss_seg, loss_adv_G, loss_D_source, loss_D_target) as device scalars."""
    H, W = images.shape[2:]
    optimizer.zero_grad()
    optimizer_D.zero_grad()
    model.train()
    model_D.train()
    for p in model_D.parameters():          # train.py:207-208
        p.requires_grad = False

    # train the segmentation net on the labelled source batch (train.py:211-221)
    loss, lr_src = supervised_loss(model, images, labels)
    loss.backward()
    allreduce_grads(_opt_params(optimizer))
    optimizer.step()

    # adversarial term on the target batch, through the frozen discriminator (train.py:223-237)
    lr_tgt = model.forward_lowres(images_t)
    optimizer.zero_grad()
    p_tgt = losses.upsample_softmax(lr_tgt[0], H, W, model.n_classes, zero_border=_zb(model_D))
    d_out = model_D(p_tgt)
    loss_adv_g = losses.bce_with_logits_const(d_out, 0.0)
    (loss_adv_g * lambda_adv).backward()
    allreduce_grads(_opt_params(optimizer))
    optimizer.step()

    # train the discriminator on detached predictions (train.py:240-262)
    for p in model_D.parameters():
        p.requires_grad = True
    out_src = lr_src[0].detach()
    d_out = model_D(losses.upsample_softmax(out_src, H, W, model.n_classes, zero_border=_zb(model_D)))
    loss_d_src = losses.bce_with_logits_const(d_out, 0.0)
    loss_d_src.backward()
    allreduce_grads(_opt_params(optimizer_D))
    optimizer_D.step()

    # softmax(out_tgt) (train.py:257) is value-identical to the tensor the adversarial pass already
    # produced from the same logits (train.py:230): reuse it, detached, instead of a second 159 MB pass
    d_out = model_D(p_tgt.detach())
    loss_d_tgt = losses.bce_with_logits_const(d_out, 1.0)
    optimizer_D.zero_grad()
    loss_d_tgt.backward()
    allreduce_grads(_opt_params(optimizer_D))
    optimizer_D.step()
    return loss.detach(), loss_adv_g.detach(), loss_d_src.detach(), loss_d_tgt.detach()


def train_da_step_nni(model, model_D, optimizer, optimizer_D, images, labels, images_t, lambda_adv=0.001):
    """The adversarial iteration of ``train_nni.py`` (train_nni.py:105-163): the discriminator and
    the adversarial term work on softmax(out32), gradients of the source and target passes
    accumulate, and each optimizer steps once at the end.

    Returns (loss_seg, lambda_adv * loss_adv_G, loss_D_source, loss_D_target) as device scalars."""
    H, W = images.shape[2:]
    model.train()
    model_D.train()
    for p in model_D.parameters():          # train_nni.py:108-109
        p.requires_grad = False
    optimizer.zero_grad()
    optimizer_D.zero_grad()

    loss, lr_src = supervised_loss(model, images, labels)          # train_nni.py:118-126
    loss.backward()

    lr_tgt = model.forward_lowres(images_t)                         # train_nni.py:132-139
    d_out = model_D(losses.upsample_softmax(lr_tgt[2], H, W, model.n_classes, zero_border=_zb(model_D)))
    loss_d1 = losses.bce_with_logits_const(d_out, 0.0) * lambda_adv
    loss_d1.backward()

    for p in model_D.parameters():          # train_nni.py:141-142
        p.requires_grad = True
    out32_src = lr_src[2].detach()
    out32_tgt = lr_tgt[2].detach()
    d_out = model_D(losses.upsample_softmax(out32_src, H, W, model.n_classes, zero_border=_zb(model_D)))  # train_nni.py:147-151
    loss_d_src = losses.bce_with_logits_const(d_out, 0.0)
    loss_d_src.backward()
    d_out = model_D(losses.upsample_softmax(out32_tgt, H, W, model.n_classes, zero_border=_zb(model_D)))  # train_nni.py:153-157
    loss_d_tgt = losses.bce_with_logits_const(d_out, 1.0)
    loss_d_tgt.backward()

    allreduce_grads(_opt_params(optimizer))
    allreduce_grads(_opt_params(optimizer_D))
    optimizer.step()                        # train_nni.py:159-161
    optimizer_D.step()
    return loss.detach(), loss_d1.detach(), loss_d_src.detach(), loss_d_tgt.detach()


def train_minent_step(model, optimizer, images, labels, images_t, lambda_ent=0.001):
    """One iteration of ADVENT's MinEnt (Vu et al., CVPR 2019): the supervised loss on the labelled source
    batch plus ``lambda_ent`` times the entropy of the target predictions (``losses.upsample_entropy`` of the
    ``out`` logits at the target image size); gradients accumulate and the optimizer steps once.

    The segmentation loss is this project's three-head ``supervised_loss`` (train.py's composition), not
    ADVENT's DeepLab main + 0.1 * aux loss; only the target term and the step structure come from ADVENT.
    Returns (loss_seg, loss_ent) as device scalars, without a host sync."""
    Ht, Wt = images_t.shape[2:]
    model.train()
    optimizer.zero_grad()
    loss, _ = supervised_loss(model, images, labels)
    loss.backward()
    lr_t = model.forward_lowres(images_t)
    loss_ent = losses.upsample_entropy(lr_t[0], Ht, Wt, model.n_classes)
    (lambda_ent * loss_ent).backward()
    allreduce_grads(_opt_params(optimizer))
    optimizer.step()
    return loss.detach(), loss_ent.detach()


def train_advent_step(model, model_D, optimizer, optimizer_D, images, labels, images_t, lambda_adv=0.001):
    """One iteration of ADVENT's AdvEnt (the ``train_advent`` loop): the discriminator works on self-information
    maps (``losses.upsample_self_information`` of the ``out`` logits) instead of on the softmax.  The net is
    trained on the source loss plus ``lambda_adv`` times the adversarial term (target maps labelled as source,
    through the frozen discriminator); the discriminator then learns source maps as 0 and target maps as 1,
    each loss halved.  Gradients accumulate and each optimizer steps once, at the end.  The target map is
    reused, detached, for the discriminator, as ``train_da_step`` reuses its softmax.

    The segmentation loss is this project's three-head ``supervised_loss`` (train.py's composition), not
    ADVENT's DeepLab main + 0.1 * aux loss, and only the main output feeds the discriminator; the target terms
    and the step structure come from ADVENT.  Works with all three discriminators.
    Returns (loss_seg, loss_adv, loss_d_src, loss_d_tgt), the last two halved, as device scalars."""
    H, W = images.shape[2:]
    Ht, Wt = images_t.shape[2:]
    ncls = model.n_classes
    zb = _zb(model_D)
    optimizer.zero_grad()
    optimizer_D.zero_grad()
    model.train()
    model_D.train()
    for p in model_D.parameters():
        p.requires_grad = False

    loss, lr_src = supervised_loss(model, images, labels)
    loss.backward()

    lr_t = model.forward_lowres(images_t)
    i_t = losses.upsample_self_information(lr_t[0], Ht, Wt, ncls, zero_border=zb)
    loss_adv = losses.bce_with_logits_const(model_D(i_t), 0.0)
    (lambda_adv * loss_adv).backward()

    for p in model_D.parameters():
        p.requires_grad = True
    i_s = losses.upsample_self_information(lr_src[0].detach(), H, W, ncls, zero_border=zb)
    loss_d_src = losses.bce_with_logits_const(model_D(i_s), 0.0) / 2
    loss_d_src.backward()
    loss_d_tgt = losses.bce_with_logits_const(model_D(i_t.detach()), 1.0) / 2
    loss_d_tgt.backward()

    allreduce_grads(_opt_params(optimizer))
    allreduce_grads(_opt_params(optimizer_D))
    optimizer.step()
    optimizer_D.step()
    return loss.detach(), loss_adv.detach(), loss_d_src.detach(), loss_d_tgt.detach()


MAX_TTA_MAPS = 16      # low-resolution maps one multi-scale combine takes (csrc/msc.cu)
MAX_DENSE_BATCH = 64   # images one forward takes: the batch limit of the [N, C] dense layers
MIN_SCALED_SIDE = 64   # smallest scaled image side predict() runs the network on


def _tta_sizes(images, scales, flip):
    """The scaled sizes (int(s*H), int(s*W)) of BiSeNet's MscEval, after checking the request."""
    n, _, H, W = images.shape
    scales = tuple(scales)
    if not scales:
        raise ValueError("scales must name at least one scale")
    if any(not (math.isfinite(s) and s > 0) for s in scales):
        raise ValueError("scales must be finite and > 0, got %r" % (scales,))
    sizes = [(int(s * H), int(s * W)) for s in scales]
    small = [(s, hw) for s, hw in zip(scales, sizes) if min(hw) < MIN_SCALED_SIDE]
    if small:
        raise ValueError("scale %r gives a %dx%d image; every scaled side must be >= %d pixels"
                         % (small[0][0], small[0][1][0], small[0][1][1], MIN_SCALED_SIDE))
    if len(scales) * (2 if flip else 1) > MAX_TTA_MAPS:
        raise ValueError("%d scales%s make %d maps; at most %d are combined" % (
            len(scales), " with flip" if flip else "", len(scales) * (2 if flip else 1), MAX_TTA_MAPS))
    if flip and 2 * n > MAX_DENSE_BATCH:
        raise ValueError("flip runs 2N = %d images in one forward; at most %d fit (use batches of <= %d)"
                         % (2 * n, MAX_DENSE_BATCH, MAX_DENSE_BATCH // 2))
    return sizes


@torch.no_grad()
def predict(model, images, n_classes=None, scales=(1.0,), flip=False, pred_dtype=torch.uint8):
    """Class map ``[N, H, W]`` of a batch of fp32 NCHW images, optionally with BiSeNet's multi-scale + flip
    test-time augmentation (MscEval): for each scale s the images are resized to (int(s*H), int(s*W))
    (bilinear, align_corners=True) and, with ``flip``, mirrored along the width; the ``out`` logits of every
    run are up-sampled to H x W (mirrored runs flipped back), their softmax probabilities summed, and the
    first maximum taken.  One scale without flip is the argmax of the up-sampled logits; ``scales=(1.0,)``
    without flip is exactly the single-scale evaluation of ``eval_batch``.  ``n_classes`` None: the model's."""
    if n_classes is None:
        n_classes = model.n_classes
    if not flip and tuple(scales) == (1.0,):   # single scale: the argmax of the up-sampled logits, any image size
        model.eval()
        H, W = images.shape[2:]
        return losses.upsample_argmax(model.forward_lowres(images)[0], H, W, n_classes, pred_dtype)
    sizes = _tta_sizes(images, scales, flip)
    maps, mirrored = _scale_maps(model, images, sizes, flip)
    H, W = images.shape[2:]
    return losses.multiscale_argmax(maps, mirrored, H, W, n_classes, pred_dtype)


def _scale_maps(model, images, sizes, flip):
    """The ``out`` low-resolution maps of MscEval's runs, one forward per scaled size (N images, or 2N with
    their mirrors) -> (maps, mirrored flags)."""
    model.eval()
    N, _, H, W = images.shape
    maps, mirrored = [], []
    for h, w in sizes:
        x = images
        if (h, w) != (H, W) or flip:
            src = images.float().contiguous()
            x = torch.empty((N * (2 if flip else 1), 3, h, w), dtype=torch.float32, device=images.device)
            K.image_rescale(src, x, mirror=flip)
        lr = model.forward_lowres(x)[0]    # a new buffer per forward: every scale's map stays valid
        maps.append(lr[:N])
        mirrored.append(False)
        if flip:
            maps.append(lr[N:])
            mirrored.append(True)
    return maps, mirrored


@torch.no_grad()
def predict_confidence(model, images, n_classes=None, scales=(1.0,), flip=False):
    """(pred uint8 [N, H, W], conf fp32 [N, H, W]) of a batch of fp32 NCHW images: ``predict``'s class map
    (same scales, flip and request checks) and each pixel's confidence, the mean over the runs of the softmax
    probability of its class.  One scale without flip: the softmax of the up-sampled logits at the argmax.
    The per-pixel input of ``pseudo_label_thresholds`` / ``pseudo_labels``.  ``n_classes`` None: the model's."""
    if n_classes is None:
        n_classes = model.n_classes
    N, _, H, W = images.shape
    # one scale without flip accepts any image size, as predict does
    sizes = [(H, W)] if not flip and tuple(scales) == (1.0,) else _tta_sizes(images, scales, flip)
    maps, mirrored = _scale_maps(model, images, sizes, flip)
    pred = torch.empty((N, H, W), dtype=torch.uint8, device=images.device)
    conf = torch.empty((N, H, W), dtype=torch.float32, device=images.device)
    K.msc_confidence([m.detach() for m in maps], mirrored, H, W, n_classes, pred, conf)
    return pred, conf


MAX_SELECT_PIXELS = 1 << 30   # pixels per selection / apply launch (csrc/pseudo.cu); larger batches are split


def _check_fraction(name, v):
    if not (isinstance(v, (int, float)) and math.isfinite(v) and 0 < v <= 1):
        raise ValueError("%s must be a finite number in (0, 1], got %r" % (name, v))


def _check_classes(n_classes):
    if not (isinstance(n_classes, int) and 2 <= n_classes <= 32):
        raise ValueError("n_classes must be an int from 2 to 32, got %r" % (n_classes,))


def _flat_chunks(*tensors):
    """Views of contiguous tensors of one shape, flattened and split into runs of <= MAX_SELECT_PIXELS."""
    flat = [t.reshape(-1) for t in tensors]
    total = flat[0].numel()
    for a in range(0, total, MAX_SELECT_PIXELS):
        yield [f[a:a + MAX_SELECT_PIXELS] for f in flat]


@torch.no_grad()
def pseudo_label_thresholds(preds, confs, n_classes=None, portion=0.5, cap=0.9):
    """Class-balanced pseudo-label thresholds (BDL's SSL stage, CBST): for each class c, the confidence at the
    top ``portion`` of the pixels predicted as c, capped at ``cap``.  Exactly: with count_c the pixels of
    class c (pred == c, conf not NaN) and k_c = min(count_c, max(1, ceil(portion * count_c))), thr_c =
    min(k_c-th largest confidence of class c, cap) in fp32; cap for a class no pixel predicts.

    ``preds`` / ``confs``: lists of per-batch tensors (uint8 / fp32 of one shape, as ``predict_confidence``
    returns them), so a whole target set can be held at 5 bytes per pixel; they are not concatenated.  Under
    torchrun each rank passes its shard (at least one batch) and every rank gets the thresholds of the union.
    ``n_classes`` None: 19 (Cityscapes / GTA5).  Returns (thr fp32 [n], counts int64 [n]) on the device,
    without a host sync."""
    n_classes = 19 if n_classes is None else n_classes
    _check_classes(n_classes)
    _check_fraction("portion", portion)
    _check_fraction("cap", cap)
    preds, confs = list(preds), list(confs)
    if not preds or len(preds) != len(confs):
        raise ValueError("preds and confs must be lists of equal, non-zero length, got %d and %d"
                         % (len(preds), len(confs)))
    for i, (p, c) in enumerate(zip(preds, confs)):
        if p.dtype != torch.uint8 or c.dtype != torch.float32 or p.shape != c.shape:
            raise ValueError("batch %d: pred must be uint8 and conf fp32 of one shape, got %s %s and %s %s"
                             % (i, p.dtype, tuple(p.shape), c.dtype, tuple(c.shape)))
    dev = preds[0].device
    state = torch.empty(3 * n_classes, dtype=torch.int64, device=dev)
    hist = torch.zeros(n_classes * 256, dtype=torch.int64, device=dev)
    thr = torch.empty(n_classes, dtype=torch.float32, device=dev)
    counts = torch.empty(n_classes, dtype=torch.int64, device=dev)
    batches = [(p.contiguous(), c.contiguous()) for p, c in zip(preds, confs)]
    world = _world()
    for pass_ in range(4):
        for p, c in batches:
            for fp, fc in _flat_chunks(p, c):
                K.class_select_hist(fp, fc, n_classes, pass_, state, hist)
        if world > 1:
            dist.all_reduce(hist)
        K.class_select_pick(n_classes, pass_, float(portion), float(cap), state, hist, thr, counts)
    return thr, counts


@torch.no_grad()
def pseudo_labels(pred, conf, thresholds, dtype=torch.int64):
    """Pseudo-labels [N, H, W]: pred where conf >= thresholds[pred], 255 (ignored by the losses) elsewhere and
    where conf is NaN.  ``thresholds``: the fp32 [n] tensor of ``pseudo_label_thresholds`` (pred >= n gives
    255), or one float, a global threshold for every class (AdaptSegNet-style SSL).  ``dtype`` int64 (for
    ``train_step``) or uint8."""
    if pred.dtype != torch.uint8 or conf.dtype != torch.float32 or pred.shape != conf.shape:
        raise ValueError("pred must be uint8 and conf fp32 of one shape, got %s %s and %s %s"
                         % (pred.dtype, tuple(pred.shape), conf.dtype, tuple(conf.shape)))
    if dtype not in (torch.uint8, torch.int64):
        raise ValueError("dtype must be torch.uint8 or torch.int64, got %s" % (dtype,))
    if torch.is_tensor(thresholds):
        if thresholds.dim() != 1 or not 2 <= thresholds.numel() <= 32:
            raise ValueError("thresholds must be a [n] tensor with n from 2 to 32, got shape %s"
                             % (tuple(thresholds.shape),))
        thr = thresholds.to(device=pred.device, dtype=torch.float32).contiguous()
    else:
        if not (isinstance(thresholds, (int, float)) and math.isfinite(thresholds)):
            raise ValueError("a global threshold must be a finite number, got %r" % (thresholds,))
        thr = torch.full((32,), float(thresholds), dtype=torch.float32, device=pred.device)
    pred, conf = pred.contiguous(), conf.contiguous()
    out = torch.empty(pred.shape, dtype=dtype, device=pred.device)
    for fp, fc, fo in _flat_chunks(pred, conf, out):
        K.pseudo_label_apply(fp, fc, thr.numel(), thr, fo)
    return out


@torch.no_grad()
def eval_batch(model, images, labels, n_classes=None, hist=None, pred_dtype=torch.uint8, scales=(1.0,), flip=False):
    """Forward + fused up-sample/argmax + confusion-matrix accumulation for a whole batch, all on
    the device (train.py:30-47 handles one image at a time through the host).  ``n_classes`` None:
    the model's.  ``scales`` / ``flip``: multi-scale + flip evaluation, see ``predict``.
    Returns (hist int64 [n*n] on the device, pred [N, H, W])."""
    if n_classes is None:
        n_classes = model.n_classes
    pred = predict(model, images, n_classes, scales, flip, pred_dtype)
    lab = labels[:, 0] if labels.dim() == 4 else labels
    hist = fast_hist_device(lab.long(), pred, n_classes, hist)
    return hist, pred


def _val_batch(model, images, labels, n_classes, hist, scales=(1.0,), flip=False):
    """One evaluation batch on the device -> (hist, per-image count of pred == label, int64 [N])."""
    hist, pred = eval_batch(model, images, labels, n_classes, hist, scales=scales, flip=flip)
    lab = labels[:, 0] if labels.dim() == 4 else labels
    if lab.dtype != torch.int64:
        lab = lab.long()
    correct = torch.zeros(images.shape[0], dtype=torch.int64, device=images.device)
    K.count_equal_batched(lab, pred, correct)
    return hist, correct


def val(model, batches, n_classes=None, device=None, scales=(1.0,), flip=False):
    """Evaluation loop (train.py:24-61): (mean pixel precision, mIoU) over ``n_classes`` classes (None:
    the model's).  ``scales`` / ``flip``: multi-scale + flip evaluation of every batch (see ``predict``).

    ``batches`` yields (images, labels) CUDA tensors -- this rank's shard of the evaluation set.  The
    confusion matrix and the per-image hit counts stay on the device for the whole loop (one
    device->host copy at the end, no per-image ``.item()``); with several ranks the int64 matrix is
    summed over them (NCCL all-reduce; BASELINE config 5) and the precision is the mean over ALL ranks'
    images, so every rank returns the same pair.  An empty shard contributes a zero matrix.
    ``precision`` reproduces the reference's arithmetic: ``float(count) / float(total)`` per image
    (utils.py:151-159), then ``np.mean`` (train.py:56)."""
    if n_classes is None:
        n_classes = model.n_classes
    hist = None
    counts, totals = [], []
    # _val_batch(model, images, labels, n_classes, hist) is the per-batch seam a CPU test replaces; the
    # multi-scale arguments are only added when they ask for more than the single-scale default
    tta = {} if (tuple(scales), bool(flip)) == ((1.0,), False) else dict(scales=scales, flip=flip)
    for images, labels in batches:
        hist, correct = _val_batch(model, images, labels, n_classes, hist, **tta)
        counts.append(correct)
        totals += [int(labels[0].numel())] * int(labels.shape[0])
        device = hist.device
    if hist is None:
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        hist = torch.zeros(n_classes * n_classes, dtype=torch.int64, device=device)
    ratios = [float(c) / float(t) for c, t in zip(torch.cat(counts).tolist(), totals)] if counts else []
    psum = torch.tensor([float(np.sum(ratios)) if ratios else 0.0, float(len(ratios))], dtype=torch.float64, device=device)
    val.last_local_hist = hist.clone() if _world() > 1 else hist   # this rank's shard, before the sum over ranks
    if _world() > 1:
        dist.all_reduce(hist)
        dist.all_reduce(psum)
        precision = float(psum[0] / psum[1]) if float(psum[1]) > 0 else float("nan")
    else:
        precision = float(np.mean(ratios)) if ratios else float("nan")
    h = hist.cpu().numpy().reshape(n_classes, n_classes).astype(np.float64)
    miou_list = per_class_iu(h)
    val.last_hist = hist      # the exact int64 matrix (summed over ranks), for callers that want it
    return precision, float(np.mean(miou_list))


class GraphedStep(object):
    """A whole train step captured once into a CUDA graph and replayed.

    At B200 speeds the step is host-bound in eager mode (about a thousand launches plus the Python
    that issues them take as long as the kernels themselves), so the forward, the hand-written
    backward, the NCCL gradient all-reduces and the fused optimizer updates are recorded into ONE
    graph with static input buffers; a replay costs a single launch.  `fn(**inputs)` must be free
    of host synchronisation (train_step / train_da_step are) and is warmed up on a side stream first
    (lazy state: packed filters, momentum buffers, NCCL communicators).  Optimizers must be
    capture-safe (``fused=True``; Adam additionally ``capturable=True``).
    """

    def __init__(self, fn, example_inputs, warmup=3, optimizers=()):
        self.fn = fn
        # A replay never runs optimizer.step() on the host again.  optim.FusedSGD / FusedAdam read
        # their hyper-parameters from device memory (poly_lr_scheduler refreshes it); a torch
        # optimizer with a Python-float lr bakes the value into the captured kernels' arguments, so
        # the reference's per-epoch decay (train.py:188-189) would silently stop: refuse that.
        for opt in optimizers:
            if hasattr(opt, "refresh_hyperparameters"):
                continue
            if any(not torch.is_tensor(g["lr"]) for g in opt.param_groups):
                raise ValueError("GraphedStep: %s has a float learning rate, which a CUDA graph freezes; build it "
                                 "with lr=torch.tensor(lr) (capturable) or use optim.FusedSGD / FusedAdam"
                                 % type(opt).__name__)
        self.static = {k: v.clone() for k, v in example_inputs.items()}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):  # at least once: lazy state must exist before capture
                fn(**self.static)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.outputs = fn(**self.static)
        from . import optim
        optim.flush_pending()   # pointer tables of optim.FusedSGD / FusedAdam steps inside the graph

    @staticmethod
    def set_lr(optimizer, lr, group=0):
        """Change a learning rate so that the next replay uses it (device-resident in both cases)."""
        g = optimizer.param_groups[group]
        if torch.is_tensor(g["lr"]):
            g["lr"].fill_(lr)
        else:
            g["lr"] = lr
            optimizer.refresh_hyperparameters()

    def load(self, **inputs):
        """Copy new inputs into the graph's static buffers (device or pinned-host tensors)."""
        for k, v in inputs.items():
            self.static[k].copy_(v, non_blocking=True)

    def __call__(self, **inputs):
        if inputs:
            self.load(**inputs)
        self.graph.replay()
        return self.outputs
