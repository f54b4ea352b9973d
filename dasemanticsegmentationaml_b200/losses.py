"""Losses and logit consumers fused with the bilinear (align_corners=True) up-sampling.

Each function takes the network's LOW-resolution class logits (fp32 ``[N, h, w, 32]`` NHWC, as
returned by ``BiSeNet.forward_lowres``) and is one autograd node backed by the kernels in
``csrc/loss.cu``; the full-size logit tensor is never written unless ``upsample_logits`` is asked
for it.  Loss composition mirrors the reference:

* ``upsample_cross_entropy``  = F.interpolate(bilinear, align_corners=True) + CrossEntropyLoss(ignore_index=255)
  (model_stages.py:240-242, train.py:66,86-89,135,214-217)
* ``upsample_softmax``        = F.interpolate + F.softmax(dim=1)           (train.py:230,248,257)
* ``bce_with_logits_const``   = BCEWithLogitsLoss against zeros / ones       (train.py:173,231-232,249-250,258)
* ``upsample_ohem_cross_entropy`` = F.interpolate + OHEM_CrossEntroy_Loss    (utils.py:256-271)
* ``upsample_argmax``         = F.interpolate + reverse_one_hot per sample   (utils.py:98-122)
* ``multiscale_argmax``       = F.interpolate + softmax summed over several maps + argmax (BiSeNet's MscEval)
* ``upsample_entropy``        = F.interpolate + softmax + ADVENT's entropy_loss        (csrc/entropy.cu)
* ``upsample_self_information`` = F.interpolate + softmax + ADVENT's prob_2_entropy    (csrc/entropy.cu)
"""
import torch

from . import kernels as K
from . import ops

F32 = torch.float32
BF16 = torch.bfloat16


class _UpsampleLogits(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lr, H, W, n_classes, dtype):
        n = lr.shape[0]
        out = torch.empty((n, n_classes, H, W), dtype=dtype, device=lr.device)
        K.upsample_fwd(lr, H, W, n_classes, K.UP_LOGITS, out=out, out_flag=1 if dtype == BF16 else 0)
        ctx.save_for_backward(lr)
        ctx.meta = (H, W, n_classes)
        return out

    @staticmethod
    def backward(ctx, dout):
        (lr,) = ctx.saved_tensors
        H, W, n_classes = ctx.meta
        d_lr = ops.zeros_f32(lr.shape, lr.device)
        dout = dout.contiguous()
        if dout.dtype not in (F32, BF16):
            dout = dout.float()
        K.upsample_bwd(lr, H, W, n_classes, K.UP_LOGITS, d_lr, grad_in=dout,
                       grad_is_bf16=1 if dout.dtype == BF16 else 0)
        return d_lr, None, None, None, None


def upsample_logits(lr, H, W, n_classes=19, dtype=F32):
    """Full-size logits ``[N, n_classes, H, W]`` (NCHW) from the low-resolution map."""
    return _UpsampleLogits.apply(lr, H, W, n_classes, dtype)


# The reference trains under nn.DataParallel (train.py:145-152,497): the batch is split over the GPUs for the
# forward only and CrossEntropyLoss runs ONCE on the gathered logits, i.e. its mean is over the valid pixels
# of the GLOBAL batch (train.py:214-217).  With one process per GPU the same value needs the (loss sum,
# valid count) pair summed over ranks -- one 16-byte all-reduce per CE term -- and every rank's gradient
# scaled by world / global count, so that the AVG gradient exchange that follows yields d(global mean)/dW.
# False: each rank normalises by its own valid count (identical when every rank sees the same number of
# labelled pixels, and what a rank-local loss would do).
GLOBAL_BATCH_MEAN = True


def _dist_world():
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


class _UpsampleCE(torch.autograd.Function):
    """Training: ONE pass computes the loss and the un-normalised gradient w.r.t. the low-resolution
    logits (the interpolation + softmax of every pixel is needed for both); backward only scales it
    by grad_out / #valid.  Without grad: the forward-only kernel."""

    @staticmethod
    def forward(ctx, lr, labels, H, W, n_classes, ignore_index):
        acc = torch.zeros(2, dtype=torch.float64, device=lr.device)
        if ctx.needs_input_grad[0]:
            d_lr = ops.zeros_f32(lr.shape, lr.device)
            K.upsample_bwd(lr, H, W, n_classes, K.UP_CE, d_lr, labels=labels, ignore_index=ignore_index,
                           loss_acc=acc)
            ctx.save_for_backward(d_lr, acc)
        else:
            K.upsample_fwd(lr, H, W, n_classes, K.UP_CE, labels=labels, ignore_index=ignore_index, acc=acc)
        ctx.grad_mul = 1.0
        world = _dist_world()
        if GLOBAL_BATCH_MEAN and world > 1:
            import torch.distributed as dist
            dist.all_reduce(acc)          # (sum of losses, valid pixels) of the global batch, in place
            ctx.grad_mul = float(world)
        return (acc[0] / acc[1]).to(F32)

    @staticmethod
    def backward(ctx, g):
        d_unscaled, acc = ctx.saved_tensors
        d_lr = torch.empty_like(d_unscaled)
        K.scale_f32(d_unscaled, g.to(F32).contiguous(), acc[1:], ctx.grad_mul, d_lr)
        return d_lr, None, None, None, None, None


# torch.nn.CrossEntropyLoss raises (device-side assert) on a label outside [0, classes) other than
# ignore_index -- an un-remapped GTA5 id, a wrong label file.  The fused kernels EXCLUDE such pixels from
# the loss, the gradient and the pixel count instead of training on them; set VALIDATE_LABELS = True to
# get the reference's behaviour (an IndexError) at the price of one extra pass + host sync per call.
VALIDATE_LABELS = False


def _check_labels(labels, n, H, W, n_classes=None, ignore_index=None):
    if labels.dim() == 4 and labels.shape[1] == 1:
        labels = labels[:, 0]
    assert labels.shape == (n, H, W), "labels must be [N, H, W] (or [N, 1, H, W])"
    if labels.dtype != torch.int64:
        labels = labels.long()
    labels = labels.contiguous()
    if VALIDATE_LABELS and n_classes is not None:
        bad = (labels < 0) | (labels >= n_classes)
        if ignore_index is not None:
            bad &= labels != ignore_index
        if bool(bad.any()):
            raise IndexError("Target %d is out of bounds." % int(labels[bad][0]))
    return labels


def upsample_cross_entropy(lr, labels, n_classes=19, ignore_index=255):
    """mean over non-ignored pixels of -log softmax(upsample(lr))[label]."""
    labels = _check_labels(labels, lr.shape[0], labels.shape[-2], labels.shape[-1], n_classes, ignore_index)
    H, W = labels.shape[1:]
    return _UpsampleCE.apply(lr, labels, H, W, n_classes, ignore_index)


class _UpsampleSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lr, H, W, n_classes, zero_border):
        n = lr.shape[0]
        if zero_border:
            # [N, H+2, W+2, 32] with the map at rows / cols 1..H / 1..W; the kernel writes the zero border
            p = torch.empty((n, H + 2, W + 2, 32), dtype=BF16, device=lr.device)
            K.upsample_fwd(lr, H, W, n_classes, K.UP_SOFTMAX, out=p, out_flag=2, p_ld=32)
            p = p[:, 1:H + 1, 1:W + 1]
        else:
            p = torch.empty((n, H, W, 32), dtype=BF16, device=lr.device)
            K.upsample_fwd(lr, H, W, n_classes, K.UP_SOFTMAX, out=p, p_ld=32)
        ctx.save_for_backward(lr)
        ctx.meta = (H, W, n_classes)
        return p.permute(0, 3, 1, 2)[:, :n_classes]

    @staticmethod
    def backward(ctx, dp):
        (lr,) = ctx.saved_tensors
        H, W, n_classes = ctx.meta
        from .model._glue import padded_base, padded_strides, to_nhwc
        d_lr = ops.zeros_f32(lr.shape, lr.device)
        if padded_strides(dp):   # the dense discriminator's pair-view data gradient: read it where it lies
            K.upsample_bwd(lr, H, W, n_classes, K.UP_SOFTMAX, d_lr, grad_in=padded_base(dp), grad_is_bf16=2, p_ld=32)
        else:
            d = to_nhwc(dp)
            K.upsample_bwd(lr, H, W, n_classes, K.UP_SOFTMAX, d_lr, grad_in=d, grad_is_bf16=1, p_ld=d.stride(2))
        return d_lr, None, None, None, None


def upsample_softmax(lr, H, W, n_classes=19, zero_border=False):
    """softmax(upsample(lr), dim=1) as a bf16 channels-last ``[N, n_classes, H, W]`` tensor (a view of
    a 32-channel NHWC buffer whose padding channels are zero) — the discriminator's input.
    zero_border=True (even H, W): the buffer is [N, H+2, W+2, 32] with a zero one-pixel border and the result
    is a ``ZeroBordered`` view of its interior; ``FCDiscriminator`` then runs its first 4x4/stride-2/pad-1 layer
    over 128-byte column pairs of that buffer (stride-1 TMA rows) instead of 64-byte stride-2 pixels.  Any other
    consumer sees an ordinary strided tensor."""
    if zero_border and H % 2 == 0 and W % 2 == 0:
        from .model._glue import ZeroBordered
        return _UpsampleSoftmax.apply(lr, H, W, n_classes, True).as_subclass(ZeroBordered)
    return _UpsampleSoftmax.apply(lr, H, W, n_classes, False)


class _UpsampleEntropy(torch.autograd.Function):
    """Training: ONE pass computes the entropy sum and the gradient of that sum w.r.t. the low-resolution
    logits (as _UpsampleCE); backward only scales it by grad_out / (N*H*W).  Without grad: the forward-only
    kernel."""

    @staticmethod
    def forward(ctx, lr, H, W, n_classes):
        acc = torch.zeros(1, dtype=torch.float64, device=lr.device)
        if ctx.needs_input_grad[0]:
            d_lr = ops.zeros_f32(lr.shape, lr.device)
            K.entropy_bwd(lr, H, W, n_classes, K.ENT_TRAIN, d_lr, acc=acc)
            ctx.save_for_backward(d_lr)
        else:
            K.entropy_fwd(lr, H, W, n_classes, K.ENT_SUM, acc=acc)
        count = lr.shape[0] * H * W
        ctx.grad_mul = 1.0 / count
        return (acc[0] / count).to(F32)

    @staticmethod
    def backward(ctx, g):
        (d_unscaled,) = ctx.saved_tensors
        d_lr = torch.empty_like(d_unscaled)
        K.scale_f32(d_unscaled, g.to(F32).contiguous(), None, ctx.grad_mul, d_lr)
        return d_lr, None, None, None


def upsample_entropy(lr, H, W, n_classes=19):
    """ADVENT's entropy loss (``entropy_loss(softmax(interp(pred)))``): the mean over the N x H x W pixels of
    the normalised entropy sum_c -p_c log p_c / log n_classes of p = softmax(upsample(lr)), an fp32 scalar.
    Nothing of size N x n x H x W is written.  Under torchrun this is the rank-local mean; the gradient average
    of ``train.allreduce_grads`` then yields the gradient of the global mean when every rank has the same batch
    shape (as ``train.train_minent_step`` is used), so no collective is needed here."""
    K.check_entropy_args(lr, H, W, n_classes)
    return _UpsampleEntropy.apply(lr, H, W, n_classes)


def _map32(d):
    """A logical bf16 [N, C, H, W] gradient as the [N, H, W, 32] NHWC buffer the self-information backward reads:
    the tensor's own storage when it is laid out so, else a copy (its channels >= C are never read)."""
    n, c, h, w = d.shape
    v = d.detach().as_subclass(torch.Tensor).permute(0, 2, 3, 1)
    if (v.dtype == BF16 and v.stride() == (h * w * 32, w * 32, 32, 1) and v.data_ptr() % 16 == 0
            and v.storage_offset() + n * h * w * 32 <= v.untyped_storage().nbytes() // 2):
        return torch.Tensor.as_strided(v, (n, h, w, 32), (h * w * 32, w * 32, 32, 1))
    buf = torch.zeros((n, h, w, 32), dtype=BF16, device=d.device)
    buf[..., :c].copy_(v)
    return buf


class _UpsampleSelfInformation(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lr, H, W, n_classes, zero_border):
        n = lr.shape[0]
        if zero_border:
            # [N, H+2, W+2, 32] with the map at rows / cols 1..H / 1..W; the kernel writes the zero border
            m = torch.empty((n, H + 2, W + 2, 32), dtype=BF16, device=lr.device)
            K.entropy_fwd(lr, H, W, n_classes, K.ENT_MAP, emap=m, layout=K.MAP_ZERO_BORDERED)
            m = m[:, 1:H + 1, 1:W + 1]
        else:
            m = torch.empty((n, H, W, 32), dtype=BF16, device=lr.device)
            K.entropy_fwd(lr, H, W, n_classes, K.ENT_MAP, emap=m, layout=K.MAP_PLAIN)
        ctx.save_for_backward(lr)
        ctx.meta = (H, W, n_classes)
        return m.permute(0, 3, 1, 2)[:, :n_classes]

    @staticmethod
    def backward(ctx, dm):
        (lr,) = ctx.saved_tensors
        H, W, n_classes = ctx.meta
        from .model._glue import padded_base, padded_strides
        d_lr = ops.zeros_f32(lr.shape, lr.device)
        if padded_strides(dm):   # the dense discriminator's pair-view data gradient: read it where it lies
            K.entropy_bwd(lr, H, W, n_classes, K.ENT_SELF_INFO, d_lr, d_map=padded_base(dm),
                          layout=K.MAP_ZERO_BORDERED)
        else:
            K.entropy_bwd(lr, H, W, n_classes, K.ENT_SELF_INFO, d_lr, d_map=_map32(dm), layout=K.MAP_PLAIN)
        return d_lr, None, None, None, None


def upsample_self_information(lr, H, W, n_classes=19, zero_border=False):
    """ADVENT's self-information map (``prob_2_entropy(softmax(interp(pred)))``): -p_c log p_c / log n_classes
    of p = softmax(upsample(lr)) as a bf16 channels-last ``[N, n_classes, H, W]`` view of a 32-channel NHWC
    buffer whose padding channels are zero -- the AdvEnt discriminator's input.  zero_border=True with even H
    and W: a ``ZeroBordered`` view of the interior of an [N, H+2, W+2, 32] buffer with a zero border, which
    ``FCDiscriminator`` reads as column pairs; otherwise a plain view (exactly as ``upsample_softmax``)."""
    K.check_entropy_args(lr, H, W, n_classes)
    if zero_border and H % 2 == 0 and W % 2 == 0:
        from .model._glue import ZeroBordered
        return _UpsampleSelfInformation.apply(lr, H, W, n_classes, True).as_subclass(ZeroBordered)
    return _UpsampleSelfInformation.apply(lr, H, W, n_classes, False)


class _BCEConst(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, target):
        xf = x.contiguous()
        out = torch.zeros((), dtype=F32, device=x.device)
        K.bce_const_fwd(xf, float(target), out)
        ctx.save_for_backward(xf)
        ctx.target = float(target)
        return out

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        dx = torch.empty_like(x)
        K.bce_const_bwd(x, ctx.target, g.to(F32).contiguous(), 1.0, dx)
        return dx, None


def bce_with_logits_const(logits, target):
    """BCEWithLogitsLoss(logits, full_like(logits, target)) for fp32 discriminator outputs."""
    assert logits.dtype == F32
    return _BCEConst.apply(logits, target)


class _UpsampleOhemCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lr, labels, H, W, n_classes, threshold, keep_num):
        n = lr.shape[0]
        dev = lr.device
        loss_map = torch.empty((n, H, W), dtype=F32, device=dev)
        acc = torch.zeros(2, dtype=torch.float64, device=dev)
        # the reference's OHEM has no ignore_index (utils.py:261): every pixel takes part
        K.upsample_fwd(lr, H, W, n_classes, K.UP_CE, labels=labels, ignore_index=-1, acc=acc, loss_map=loss_map)
        state = torch.empty(2, dtype=torch.int32, device=dev)
        hist = torch.empty(256, dtype=torch.int32, device=dev)
        K.radix_select_desc(loss_map, keep_num, state, hist)
        sums = torch.empty(5, dtype=torch.float64, device=dev)
        sel = torch.empty(4, dtype=F32, device=dev)
        K.ohem_reduce(loss_map, state, threshold, keep_num, sums, sel)
        ctx.save_for_backward(lr, labels, loss_map, sel)
        ctx.meta = (H, W, n_classes)
        return sel[0].clone()

    @staticmethod
    def backward(ctx, g):
        lr, labels, loss_map, sel = ctx.saved_tensors
        H, W, n_classes = ctx.meta
        weights = torch.empty_like(loss_map)
        K.ohem_weights(loss_map, sel, weights)
        d_lr = ops.zeros_f32(lr.shape, lr.device)
        K.upsample_bwd(lr, H, W, n_classes, K.UP_CE, d_lr, labels=labels, ignore_index=-1,
                       pixel_weight=weights, coef_num=g.to(F32).contiguous())
        return d_lr, None, None, None, None, None, None


def upsample_ohem_cross_entropy(lr, labels, threshold, keep_num, n_classes=19):
    """OHEM_CrossEntroy_Loss(threshold, keep_num)(upsample(lr), labels) with a radix-select k-th
    largest instead of torch.sort.  Labels must lie in [0, n_classes): the reference raises otherwise; here such
    pixels contribute a zero loss (see VALIDATE_LABELS)."""
    labels = _check_labels(labels, lr.shape[0], labels.shape[-2], labels.shape[-1], n_classes, None)
    H, W = labels.shape[1:]
    if not (0 <= keep_num < labels.numel()):
        raise IndexError("keep_num %d out of range for %d pixels" % (keep_num, labels.numel()))
    return _UpsampleOhemCE.apply(lr, labels, H, W, n_classes, float(threshold), int(keep_num))


def upsample_argmax(lr, H, W, n_classes=19, dtype=torch.int64):
    """Per-pixel class map ``[N, H, W]`` (int64 like reverse_one_hot, or uint8)."""
    n = lr.shape[0]
    out = torch.empty((n, H, W), dtype=dtype, device=lr.device)
    with torch.no_grad():
        K.upsample_fwd(lr.detach(), H, W, n_classes, K.UP_ARGMAX, out=out, out_flag=1 if dtype == torch.uint8 else 0)
    return out


def multiscale_argmax(maps, mirrored, H, W, n_classes=19, dtype=torch.int64):
    """argmax over classes of sum_k softmax(upsample(maps[k])) ``[N, H, W]``, each mirrored map's up-sampled
    probabilities flipped back along the width (BiSeNet's MscEval combine).  One unmirrored map: softmax does
    not move the argmax, so this is ``upsample_argmax``."""
    if len(maps) == 1 and not mirrored[0]:
        return upsample_argmax(maps[0], H, W, n_classes, dtype)
    out = torch.empty((maps[0].shape[0], H, W), dtype=dtype, device=maps[0].device)
    with torch.no_grad():
        K.msc_argmax([m.detach() for m in maps], mirrored, H, W, n_classes, out)
    return out
