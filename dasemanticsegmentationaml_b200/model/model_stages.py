"""BiSeNet (STDC) on the B200 kernels — drop-in for the reference's ``model/model_stages.py``.

Same class names, constructor signatures, ``forward`` returns, ``get_params`` grouping and
state_dict keys.  What changes is below the module API:

* ContextPath / FFM / heads are composed from fused kernels with a hand-written backward
  (one autograd node per module call, no per-op autograd graph);
* the global-pool attention vectors ([N, C]) run through tiny fp32 kernels; the per-pixel
  scale / add / nearest-upsample steps (model_stages.py:85,123,126-127,131-132,183-184) are one
  pass each;
* ``torch.cat`` of the FFM (model_stages.py:176) is replaced by having its two producers write
  into one 384-channel buffer;
* ``BiSeNet.forward_lowres`` exposes the 1/8- and 1/16-resolution logits so that the losses can
  fuse the bilinear up-sampling (see losses.py); ``forward`` still returns full-size logits.
"""
import numbers

import torch
import torch.nn as nn

from .. import kernels as K
from .. import ops
from ._glue import B200Module, bn_tuple, run_module, to_nhwc
from .stdcnet import STDCNet813

BatchNorm2d = nn.BatchNorm2d
F32 = torch.float32


def _kaiming_children(module):
    for ly in module.children():
        if isinstance(ly, nn.Conv2d):
            nn.init.kaiming_normal_(ly.weight, a=1)
            if ly.bias is not None:
                nn.init.constant_(ly.bias, 0)


def _wd_groups(module):
    """get_params of the reference (model_stages.py:55-65 and siblings)."""
    wd_params, nowd_params = [], []
    for name, m in module.named_modules():
        if isinstance(m, (nn.Linear, nn.Conv2d)):
            wd_params.append(m.weight)
            if m.bias is not None:
                nowd_params.append(m.bias)
        elif isinstance(m, BatchNorm2d):
            nowd_params += list(m.parameters())
    return wd_params, nowd_params


class ConvBNReLU(B200Module):
    """conv(ks, stride, padding, bias=False) -> BatchNorm2d -> ReLU (reference model_stages.py:11-35)."""

    def __init__(self, in_chan, out_chan, ks=3, stride=1, padding=1, *args, **kwargs):
        super(ConvBNReLU, self).__init__()
        self.conv = nn.Conv2d(in_chan, out_chan, kernel_size=ks, stride=stride, padding=padding, bias=False)
        self.bn = BatchNorm2d(out_chan)
        self.relu = nn.ReLU()
        self.init_weight()

    def init_weight(self):
        _kaiming_children(self)

    def _fwd(self, x, out=None):
        return ops.conv_bn_act_fwd(x, self.conv.weight, bn_tuple(self.bn, self.training),
                                   self.conv.stride[0], self.conv.padding[0], self.training,
                                   K.ACT_RELU, out=out)

    def _bwd(self, ctx, dy1, dy2=None, need_dx=True):
        dx, dw, dg, db = ops.conv_bn_act_bwd(ctx, dy1, dy2, need_dx)
        return dx, {self.conv.weight: dw, self.bn.weight: dg, self.bn.bias: db}

    # [N, C, 1, 1] inputs (conv_avg after the global pool) go through the dense-vector kernels
    def _fwd_vec(self, pooled_sum, in_scale):
        assert self.conv.kernel_size == (1, 1)
        return ops.fc_fwd(pooled_sum, in_scale, self.conv.weight, bn_tuple(self.bn, self.training),
                          self.training, K.ACT_RELU)

    def _bwd_vec(self, ctx, dout):
        din, dw, dg, db = ops.fc_bwd(ctx, dout)
        return din, {self.conv.weight: dw, self.bn.weight: dg, self.bn.bias: db}


# Class counts the fused up-sampling losses are compiled for (csrc/loss.cu): the logits are 32 floats per pixel.
MIN_CLASSES, MAX_CLASSES = 2, 32
LOGIT_CHANNELS = 32
# The class heads' weight-gradient tiles in tuned_tiles.json were swept at 19 classes.  The tile fixes
# the reduction (Cin) tiling and the pixel split; every count up to 32 is one output-row tile, so every
# count uses the same entries.
TUNED_HEAD_CLASSES = 19


def check_n_classes(n_classes):
    if not (isinstance(n_classes, numbers.Integral) and not isinstance(n_classes, bool)
            and MIN_CLASSES <= n_classes <= MAX_CLASSES):
        raise ValueError("n_classes must be an integer from %d to %d (the compiled class counts), got %r"
                         % (MIN_CLASSES, MAX_CLASSES, n_classes))


class BiSeNetOutput(B200Module):
    """ConvBNReLU 3x3 -> 1x1 conv to n_classes (reference model_stages.py:38-65).
    Internally the class logits are fp32 NHWC, 32 channels whatever n_classes (2..32): the 1x1 filter
    is packed as 32 rows, rows >= n_classes zero, so every class count runs the 19-class head's
    shapes and tuned tiles."""

    def __init__(self, in_chan, mid_chan, n_classes, *args, **kwargs):
        check_n_classes(n_classes)
        super(BiSeNetOutput, self).__init__()
        self.conv = ConvBNReLU(in_chan, mid_chan, ks=3, stride=1, padding=1)
        self.conv_out = nn.Conv2d(mid_chan, n_classes, kernel_size=1, bias=False)
        self.init_weight()

    def init_weight(self):
        _kaiming_children(self)

    def get_params(self):
        return _wd_groups(self)

    def _fwd(self, x):
        mid, c = self.conv._fwd(x)
        logits = ops.conv_raw_fwd(mid, self.conv_out.weight, 1, 0, out_dtype=F32, rows_pad=LOGIT_CHANNELS)
        return logits, {"conv": c, "mid": mid}

    def _bwd(self, ctx, d_logits, need_dx=True):
        """d_logits: fp32 [N, h, w, 32] (contiguous)."""
        dz = torch.empty(d_logits.shape, dtype=torch.bfloat16, device=d_logits.device)
        K.cast_f32_bf16(d_logits, dz)
        mid = ctx["mid"]
        ncls = self.conv_out.weight.shape[0]
        dw_out = ops.conv_wgrad(dz[..., :ncls], mid, self.conv_out.weight, 1, 0, tune_cout=TUNED_HEAD_CLASSES)
        d_mid = ops.conv_dgrad(dz, self.conv_out.weight, 1, 0, mid.shape[1], mid.shape[2])
        dx, g = self.conv._bwd(ctx["conv"], d_mid, None, need_dx)
        g[self.conv_out.weight] = dw_out
        return dx, g

    def _fwd_api(self, x):
        logits, ctx = self._fwd(to_nhwc(x))
        ncls = self.conv_out.weight.shape[0]
        return logits[..., :ncls].permute(0, 3, 1, 2), ctx

    def _bwd_api(self, ctx, dout, need_dx=True, need_dw=True):
        n, c, h, w = dout.shape
        d = ops.zeros_f32((n, h, w, LOGIT_CHANNELS), dout.device)
        d[..., :c].copy_(dout.permute(0, 2, 3, 1))
        dx, g = self._bwd(ctx, d, need_dx)
        return (None if dx is None else dx.permute(0, 3, 1, 2)), g


class AttentionRefinementModule(B200Module):
    """ConvBNReLU 3x3 -> global pool -> 1x1 conv -> BN -> sigmoid -> feat * atten
    (reference model_stages.py:68-91)."""

    def __init__(self, in_chan, out_chan, *args, **kwargs):
        super(AttentionRefinementModule, self).__init__()
        self.conv = ConvBNReLU(in_chan, out_chan, ks=3, stride=1, padding=1)
        self.conv_atten = nn.Conv2d(out_chan, out_chan, kernel_size=1, bias=False)
        self.bn_atten = BatchNorm2d(out_chan)
        self.sigmoid_atten = nn.Sigmoid()
        self.init_weight()

    def init_weight(self):
        _kaiming_children(self)

    def _fwd_tail(self, x, add_vec=None, add_t=None, out_hw=None):
        """ARM, then ``+ add`` (a per-image vector or a same-size tensor), then nearest up-sampling
        to ``out_hw`` — the three steps of model_stages.py:125-127 / 130-132 in one pass."""
        feat, c_conv = self.conv._fwd(x)
        n, h, w, c = feat.shape
        pooled = ops.pool_sum(feat)
        att, c_fc = ops.fc_fwd(pooled, 1.0 / (h * w), self.conv_atten.weight,
                               bn_tuple(self.bn_atten, self.training), self.training, K.ACT_SIGMOID)
        ho, wo = out_hw if out_hw is not None else (h, w)
        out = ops.empty_act(n, ho, wo, c, feat.device)
        K.scale_add_bcast(feat, att, 0.0, add_vec, 1.0, add_t, out)
        return out, {"conv": c_conv, "fc": c_fc, "feat": feat, "att": att, "has_vec": add_vec is not None,
                     "has_t": add_t is not None}

    def _bwd_tail(self, ctx, dout, need_dx=True):
        """-> (dx, d_add_vec [N,C] or None, d_add_t (tensor at feat size) or None, grads)"""
        feat, att = ctx["feat"], ctx["att"]
        n, h, w, c = feat.shape
        dev = feat.device
        d_att = ops.zeros_f32((n, c), dev)
        d_vec = ops.zeros_f32((n, c), dev) if ctx["has_vec"] else None
        same = dout.shape[1] == h and dout.shape[2] == w
        dsum = dout if same else ops.empty_act(n, h, w, c, dev)
        K.upsum_dot_reduce(dout, feat, None if same else dsum, h, w, d_att, d_vec)
        d_pooled, dw, dg, db = ops.fc_bwd(ctx["fc"], d_att)
        d_feat = ops.empty_act(n, h, w, c, dev)
        K.scale_add_bcast(dsum, att, 0.0, d_pooled, 1.0, None, d_feat)
        dx, g = self.conv._bwd(ctx["conv"], d_feat, None, need_dx)
        g.update({self.conv_atten.weight: dw, self.bn_atten.weight: dg, self.bn_atten.bias: db})
        return dx, d_vec, (dsum if ctx["has_t"] else None), g

    def _fwd(self, x):
        return self._fwd_tail(x)

    def _bwd(self, ctx, dout, need_dx=True):
        dx, _, _, g = self._bwd_tail(ctx, dout, need_dx)
        return dx, g


class ContextPath(B200Module):
    """Backbone + ARM16/ARM32 + global-average branch + two head convs (reference model_stages.py:94-152)."""

    def __init__(self, backbone='CatNetSmall', pretrain_model='', use_conv_last=False, *args, **kwargs):
        super(ContextPath, self).__init__()
        self.backbone = STDCNet813(pretrain_model=pretrain_model, use_conv_last=use_conv_last)
        self.arm16 = AttentionRefinementModule(512, 128)
        inplanes = 1024
        self.arm32 = AttentionRefinementModule(inplanes, 128)
        self.conv_head32 = ConvBNReLU(128, 128, ks=3, stride=1, padding=1)
        self.conv_head16 = ConvBNReLU(128, 128, ks=3, stride=1, padding=1)
        self.conv_avg = ConvBNReLU(inplanes, 128, ks=1, stride=1, padding=0)
        self.init_weight()

    def init_weight(self):
        _kaiming_children(self)

    def get_params(self):
        return _wd_groups(self)

    def _fwd(self, img, feat8_out=None, cp8_out=None):
        (feat2, feat4, feat8, feat16, feat32), c_bb = self.backbone._fwd(img, feat8_out=feat8_out)
        h8, w8 = feat8.shape[1:3]
        h16, w16 = feat16.shape[1:3]
        h32, w32 = feat32.shape[1:3]
        pooled32 = ops.pool_sum(feat32)
        avg, c_avg = self.conv_avg._fwd_vec(pooled32, 1.0 / (h32 * w32))
        up32, c_arm32 = self.arm32._fwd_tail(feat32, add_vec=avg, out_hw=(h16, w16))
        feat32_up, c_h32 = self.conv_head32._fwd(up32)
        up16, c_arm16 = self.arm16._fwd_tail(feat16, add_t=feat32_up, out_hw=(h8, w8))
        feat16_up, c_h16 = self.conv_head16._fwd(up16, out=cp8_out)
        ctx = {"bb": c_bb, "avg": c_avg, "arm32": c_arm32, "h32": c_h32, "arm16": c_arm16, "h16": c_h16,
               "shape32": feat32.shape}
        return (feat2, feat4, feat8, feat16, feat16_up, feat32_up), ctx

    def _bwd(self, ctx, d2=None, d4=None, d8=None, d16=None, d_cp8=None, d_cp16=None, need_dx=False,
             d_cp8_b=None):
        grads = {}
        d16_arm = d32_int = None
        if d_cp8 is not None or d_cp8_b is not None:
            a, b = (d_cp8, d_cp8_b) if d_cp8 is not None else (d_cp8_b, None)
            d_up16, g = self.conv_head16._bwd(ctx["h16"], a, b, True)
            grads.update(g)
            d16_arm, _, d32_int, g = self.arm16._bwd_tail(ctx["arm16"], d_up16, True)
            grads.update(g)
        d32_arm = None
        if d_cp16 is not None or d32_int is not None:
            a, b = (d_cp16, d32_int) if d_cp16 is not None else (d32_int, None)
            d_up32, g = self.conv_head32._bwd(ctx["h32"], a, b, True)
            grads.update(g)
            d32_arm, d_avg, _, g = self.arm32._bwd_tail(ctx["arm32"], d_up32, True)
            grads.update(g)
            d_pooled32, g = self.conv_avg._bwd_vec(ctx["avg"], d_avg)
            grads.update(g)
            d32_arm = ops.add_bcast_vec(d32_arm, d_pooled32)
        d16_tot = d16_arm if d16 is None else (d16 if d16_arm is None else ops.add_acts(d16, d16_arm))
        _, g = self.backbone._bwd(ctx["bb"], d2, d4, d8, d16_tot, d32_arm)
        grads.update(g)
        return None, grads

    def _fwd_api(self, x):
        feats, ctx = self._fwd(x.float().contiguous())
        return tuple(f.permute(0, 3, 1, 2) for f in feats), ctx


class FeatureFusionModule(B200Module):
    """cat -> ConvBNReLU 1x1 -> global pool -> 1x1 -> ReLU -> 1x1 -> sigmoid -> feat*att + feat
    (reference model_stages.py:155-202)."""

    def __init__(self, in_chan, out_chan, *args, **kwargs):
        super(FeatureFusionModule, self).__init__()
        self.convblk = ConvBNReLU(in_chan, out_chan, ks=1, stride=1, padding=0)
        self.conv1 = nn.Conv2d(out_chan, out_chan // 4, kernel_size=1, stride=1, padding=0, bias=False)
        self.conv2 = nn.Conv2d(out_chan // 4, out_chan, kernel_size=1, stride=1, padding=0, bias=False)
        self.relu = nn.ReLU(inplace=True)
        self.sigmoid = nn.Sigmoid()
        self.init_weight()

    def init_weight(self):
        _kaiming_children(self)

    def get_params(self):
        return _wd_groups(self)

    def _fwd_cat(self, fcat):
        feat, c_blk = self.convblk._fwd(fcat)
        n, h, w, c = feat.shape
        pooled = ops.pool_sum(feat)
        a1, c1 = ops.fc_fwd(pooled, 1.0 / (h * w), self.conv1.weight, None, self.training, K.ACT_RELU)
        att, c2 = ops.fc_fwd(a1, 1.0, self.conv2.weight, None, self.training, K.ACT_SIGMOID)
        out = ops.empty_act(n, h, w, c, feat.device)
        K.scale_add_bcast(feat, att, 1.0, None, 0.0, None, out)
        return out, {"blk": c_blk, "fc1": c1, "fc2": c2, "feat": feat, "att": att}

    def _bwd_cat(self, ctx, dout, need_dx=True):
        feat, att = ctx["feat"], ctx["att"]
        n, h, w, c = feat.shape
        d_att = ops.zeros_f32((n, c), feat.device)
        K.upsum_dot_reduce(dout, feat, None, h, w, d_att, None)
        d_a1, dw2, _, _ = ops.fc_bwd(ctx["fc2"], d_att)
        d_pooled, dw1, _, _ = ops.fc_bwd(ctx["fc1"], d_a1)
        d_feat = ops.empty_act(n, h, w, c, feat.device)
        K.scale_add_bcast(dout, att, 1.0, d_pooled, 1.0, None, d_feat)
        d_fcat, g = self.convblk._bwd(ctx["blk"], d_feat, None, need_dx)
        g.update({self.conv1.weight: dw1, self.conv2.weight: dw2})
        return d_fcat, g

    def _fwd(self, fsp, fcp):
        n, h, w, c1 = fsp.shape
        c2 = fcp.shape[3]
        fcat = ops.empty_act(n, h, w, c1 + c2, fsp.device)
        K.scale_add_bcast(fsp, None, 1.0, None, 0.0, None, fcat[..., :c1])
        K.scale_add_bcast(fcp, None, 1.0, None, 0.0, None, fcat[..., c1:])
        out, ctx = self._fwd_cat(fcat)
        ctx["split"] = c1
        return out, ctx

    def _bwd(self, ctx, dout, need_dx=True):
        d_fcat, g = self._bwd_cat(ctx, dout, need_dx)
        c1 = ctx["split"]
        return (d_fcat[..., :c1], d_fcat[..., c1:]), g


class BiSeNet(B200Module):
    """BiSeNet with the STDC backbone (reference model_stages.py:205-270)."""

    def __init__(self, backbone, n_classes, pretrain_model='', use_boundary_2=False, use_boundary_4=False,
                 use_boundary_8=False, use_boundary_16=False, use_conv_last=False, heat_map=False, *args, **kwargs):
        check_n_classes(n_classes)
        super(BiSeNet, self).__init__()
        self.cp = ContextPath(backbone, pretrain_model, use_conv_last=use_conv_last)
        conv_out_inplanes = 128
        sp8_inplanes = 256
        inplane = sp8_inplanes + conv_out_inplanes
        self.ffm = FeatureFusionModule(inplane, 256)
        self.conv_out = BiSeNetOutput(256, 256, n_classes)
        self.conv_out16 = BiSeNetOutput(conv_out_inplanes, 64, n_classes)
        self.conv_out32 = BiSeNetOutput(conv_out_inplanes, 64, n_classes)
        self.n_classes = n_classes
        self.logits_dtype = torch.float32  # dtype of the full-size logits returned by forward()
        if ".pth" not in pretrain_model:
            self.init_weight()
        else:
            self.load_weight(pretrain_model)

    def init_weight(self):
        _kaiming_children(self)

    def load_weight(self, pretrain_model):
        state_dict = torch.load(pretrain_model)
        own = self.state_dict()
        for k, v in state_dict.items():
            own.update({k: v})
        self.load_state_dict(own)

    def get_params(self):
        wd_params, nowd_params, lr_mul_wd_params, lr_mul_nowd_params = [], [], [], []
        for name, child in self.named_children():
            child_wd_params, child_nowd_params = child.get_params()
            if isinstance(child, (FeatureFusionModule, BiSeNetOutput)):
                lr_mul_wd_params += child_wd_params
                lr_mul_nowd_params += child_nowd_params
            else:
                wd_params += child_wd_params
                nowd_params += child_nowd_params
        return wd_params, nowd_params, lr_mul_wd_params, lr_mul_nowd_params

    # -- low-resolution composite -------------------------------------------------------------
    def _fwd(self, img):
        n, _, H, W = img.shape
        h8, w8 = ((H - 1) // 2 + 1), ((W - 1) // 2 + 1)
        for _ in range(2):
            h8, w8 = (h8 - 1) // 2 + 1, (w8 - 1) // 2 + 1
        fcat = ops.empty_act(n, h8, w8, 384, img.device)
        feats, c_cp = self.cp._fwd(img, feat8_out=fcat[..., :256], cp8_out=fcat[..., 256:])
        feat_cp8, feat_cp16 = feats[4], feats[5]
        fuse, c_ffm = self.ffm._fwd_cat(fcat)
        lr_out, c1 = self.conv_out._fwd(fuse)
        lr16, c2 = self.conv_out16._fwd(feat_cp8)
        lr32, c3 = self.conv_out32._fwd(feat_cp16)
        return (lr_out, lr16, lr32), {"cp": c_cp, "ffm": c_ffm, "o": c1, "o16": c2, "o32": c3}

    def _bwd(self, ctx, d_out=None, d_out16=None, d_out32=None, need_dx=False):
        grads = {}
        d_feat8 = d_cp8 = d_cp8_b = d_cp16 = None
        if d_out is not None:
            d_fuse, g = self.conv_out._bwd(ctx["o"], d_out)
            grads.update(g)
            d_fcat, g = self.ffm._bwd_cat(ctx["ffm"], d_fuse)
            grads.update(g)
            d_feat8, d_cp8 = d_fcat[..., :256], d_fcat[..., 256:]
        if d_out16 is not None:
            d_cp8_b, g = self.conv_out16._bwd(ctx["o16"], d_out16)
            grads.update(g)
        if d_out32 is not None:
            d_cp16, g = self.conv_out32._bwd(ctx["o32"], d_out32)
            grads.update(g)
        _, g = self.cp._bwd(ctx["cp"], None, None, d_feat8, None, d_cp8, d_cp16, d_cp8_b=d_cp8_b)
        grads.update(g)
        return None, grads

    def _fwd_api(self, x):
        return self._fwd(x.float().contiguous())

    def _bwd_api(self, ctx, *douts, need_dx=False, need_dw=True):
        ds = [None if d is None else d.contiguous() for d in douts]
        return self._bwd(ctx, *ds)

    def forward_lowres(self, x):
        """The three class-logit maps before up-sampling: fp32 ``[N, h, w, 32]`` (NHWC, classes
        padded to 32) at 1/8, 1/8 and 1/16 resolution.  Feed them to the fused losses."""
        return run_module(self, x)

    def forward(self, x):
        from ..losses import upsample_logits
        H, W = x.shape[2:]
        lr = self.forward_lowres(x)
        return tuple(upsample_logits(t, H, W, self.n_classes, self.logits_dtype) for t in lr)
