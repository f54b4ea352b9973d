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
import numpy as np
import torch
import torch.distributed as dist

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


@torch.no_grad()
def eval_batch(model, images, labels, n_classes=None, hist=None, pred_dtype=torch.uint8):
    """Forward + fused up-sample/argmax + confusion-matrix accumulation for a whole batch, all on
    the device (train.py:30-47 handles one image at a time through the host).  ``n_classes`` None:
    the model's.  Returns (hist int64 [n*n] on the device, pred [N, H, W])."""
    if n_classes is None:
        n_classes = model.n_classes
    model.eval()
    H, W = images.shape[2:]
    lr = model.forward_lowres(images)
    pred = losses.upsample_argmax(lr[0], H, W, n_classes, pred_dtype)
    lab = labels[:, 0] if labels.dim() == 4 else labels
    hist = fast_hist_device(lab.long(), pred, n_classes, hist)
    return hist, pred


def _val_batch(model, images, labels, n_classes, hist):
    """One evaluation batch on the device -> (hist, per-image count of pred == label, int64 [N])."""
    from . import kernels as K
    hist, pred = eval_batch(model, images, labels, n_classes, hist)
    lab = labels[:, 0] if labels.dim() == 4 else labels
    if lab.dtype != torch.int64:
        lab = lab.long()
    correct = torch.zeros(images.shape[0], dtype=torch.int64, device=images.device)
    K.count_equal_batched(lab, pred, correct)
    return hist, correct


def val(model, batches, n_classes=None, device=None):
    """Evaluation loop (train.py:24-61): (mean pixel precision, mIoU) over ``n_classes`` classes (None:
    the model's).

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
    for images, labels in batches:
        hist, correct = _val_batch(model, images, labels, n_classes, hist)
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
