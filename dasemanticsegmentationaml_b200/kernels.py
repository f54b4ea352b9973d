"""Thin tensor-level wrappers over the C-ABI entry points of libb200seg.so.

Activations are NHWC bf16 tensors ``[N, H, W, C]`` whose innermost stride is 1; a channel slice of a
wider buffer (``buf[..., a:b]``) is passed as-is — the kernels take the pixel stride from
``stride(2)``, which is how concatenations are built without a copy.
Every function launches on the current torch stream and returns immediately.
"""
import ctypes

import torch

from . import _lib
from ._lib import c_float, c_int, c_int64, call, check, int_array, lib, ptr, stream


def round_up(v, m):
    return (v + m - 1) // m * m


def _nhwc_meta(t):
    assert t.dim() == 4 and t.stride(3) == 1, "expected an NHWC tensor with unit channel stride"
    n, h, w, c = t.shape
    ld = t.stride(2)
    assert t.stride(1) == w * ld and t.stride(0) == h * w * ld, "NHWC view must be pixel-dense"
    return n, h, w, c, ld


# ------------------------------------------------------------------ filter packing
def pack_filter(weight, transpose=False, rows_pad=None):
    """fp32 ``[Cout, Cin, R, S]`` -> bf16 ``[rows_pad, R*S, inner_pad]`` K-major GEMM operand.

    ``transpose=False``: rows = Cout (forward).  ``transpose=True``: rows = Cin (data gradient).
    rows are padded to a multiple of 16 (or to ``rows_pad``, zero rows), the inner (reduction) channel
    count to 32 or 64.
    """
    cout, cin, r, s = weight.shape
    rows, inner = (cin, cout) if transpose else (cout, cin)
    rows_pad = round_up(rows, 16) if rows_pad is None else rows_pad
    assert rows_pad >= rows and rows_pad % 16 == 0
    inner_pad = round_up(inner, 32) if inner <= 32 else round_up(inner, 64)
    out = torch.empty((rows_pad, r * s, inner_pad), dtype=torch.bfloat16, device=weight.device)
    w = weight.detach()
    if w.dtype != torch.float32 or not w.is_contiguous():
        w = w.float().contiguous()
    call("b200_pack_filter", ptr(w), ptr(out), c_int(cout), c_int(cin), c_int(r * s),
                                 c_int(rows_pad), c_int(inner_pad), c_int(1 if transpose else 0),
                                 stream())
    return out


# ------------------------------------------------------------------ geometry
class Geometry(object):
    """Tap tables of one implicit-GEMM launch, with the ctypes arrays pre-built (cached per shape)."""

    def __init__(self, classes, in_stride, out_stride, hout, wout, key=""):
        self.key = key
        self.classes, self.in_stride, self.out_stride, self.Hout, self.Wout = classes, in_stride, out_stride, hout, wout
        self.tmax = max(len(c["taps"]) for c in classes)
        flat = []
        for c in classes:
            for t in range(self.tmax):
                flat += list(c["taps"][t]) if t < len(c["taps"]) else [0, 0, 0]
        self.c_n = c_int(len(classes))
        self.c_ho = int_array([c["Ho"] for c in classes])
        self.c_wo = int_array([c["Wo"] for c in classes])
        self.c_oa = int_array([c["oa"] for c in classes])
        self.c_ob = int_array([c["ob"] for c in classes])
        self.c_nt = int_array([len(c["taps"]) for c in classes])
        self.c_taps = int_array(flat)
        self.px_taps = sum(c["Ho"] * c["Wo"] * len(c["taps"]) for c in classes)

    def __getitem__(self, key):  # dict-style access used by callers/tests
        return getattr(self, key)


_geom_cache = {}


def fwd_geometry(hin, win, r, s, stride, pad):
    key = ("f", hin, win, r, s, stride, pad)
    g = _geom_cache.get(key)
    if g is None:
        ho = (hin + 2 * pad - r) // stride + 1
        wo = (win + 2 * pad - s) // stride + 1
        taps = [(i - pad, j - pad, i * s + j) for i in range(r) for j in range(s)]
        g = _geom_cache[key] = Geometry([dict(Ho=ho, Wo=wo, oa=0, ob=0, taps=taps)], stride, 1, ho, wo,
                                        "f%dx%ds%dp%d" % (r, s, stride, pad))
    return g


def dgrad_geometry(hin, win, r, s, stride, pad):
    """Geometry of dx[N,hin,win,Cin] = conv_transpose(dz); dz is the kernel's *input*.  A stride-2
    conv splits into the four output-parity classes, each a stride-1 conv over dz with its own taps."""
    key = ("d", hin, win, r, s, stride, pad)
    g = _geom_cache.get(key)
    if g is not None:
        return g
    if stride == 1:
        taps = [(pad - i, pad - j, i * s + j) for i in range(r) for j in range(s)]
        g = Geometry([dict(Ho=hin, Wo=win, oa=0, ob=0, taps=taps)], 1, 1, hin, win,
                     "d%dx%ds%dp%d" % (r, s, stride, pad))
    else:
        assert stride == 2
        classes = []
        for a in range(2):
            for b in range(2):
                taps = [((a + pad - i) // 2, (b + pad - j) // 2, i * s + j)
                        for i in range(r) if (a + pad - i) % 2 == 0
                        for j in range(s) if (b + pad - j) % 2 == 0]
                hc, wc = (hin - a + 1) // 2, (win - b + 1) // 2
                if not taps:
                    raise ValueError("strided dgrad class without taps (1x1 stride-2 conv?)")
                if hc > 0 and wc > 0:
                    classes.append(dict(Ho=hc, Wo=wc, oa=a, ob=b, taps=taps))
        g = Geometry(classes, 1, 2, hin, win, "d%dx%ds%dp%d" % (r, s, stride, pad))
    _geom_cache[key] = g
    return g


def pairview_fwd_geometry(h, w):
    """Conv2d(k=4, s=2, p=1) over an [h, w] map stored zero-bordered as [h+2][w+2][32], seen as the
    [(h+2)/2][w+2][64] view of its column pairs (a view row = two bordered rows side by side): tap
    (a, r, b) = kernel row 2a + r, kernel columns 2b, 2b+1 reads view pixel (ho + a, r*(w+2)/2 + wo + b) --
    a stride-1 filter of 8 taps with 128-byte rows and no padding left to do."""
    key = ("pvf", h, w)
    g = _geom_cache.get(key)
    if g is None:
        assert h % 2 == 0 and w % 2 == 0
        half = (w + 2) // 2
        taps = [(a, r * half + b, (2 * a + r) * 2 + b) for a in range(2) for r in range(2) for b in range(2)]
        g = _geom_cache[key] = Geometry([dict(Ho=h // 2, Wo=w // 2, oa=0, ob=0, taps=taps)], 1, 1, h // 2, w // 2, "pvf4x4s2p1")
    return g


def pairview_dgrad_geometry(h, w):
    """Data gradient of the same layer, written straight into the pair view [(h+2)/2][w+2][64] of the
    zero-bordered gradient map: view row-half r (class r) gets the taps with kernel row parity r."""
    key = ("pvd", h, w)
    g = _geom_cache.get(key)
    if g is None:
        half = (w + 2) // 2
        classes = [dict(Ho=(h + 2) // 2, Wo=half, oa=0, ob=r * half,
                        taps=[(-a, -b, (2 * a + r) * 2 + b) for a in range(2) for b in range(2)]) for r in range(2)]
        g = _geom_cache[key] = Geometry(classes, 1, 1, (h + 2) // 2, w + 2, "pvd4x4s2p1")
    return g


# ------------------------------------------------------------------ tuned tile table
# Produced on a B200 by scripts/tune_conv.py (exhaustive sweep per layer shape); a missing key falls
# back to the launcher's heuristic.  RECORD, when a list, collects the keys a workload touches.
TUNED = {}
RECORD = None


def load_tuned(path=None):
    import json
    import os
    path = path or os.path.join(os.path.dirname(os.path.abspath(__file__)), "tuned_tiles.json")
    if os.path.exists(path):
        with open(path) as f:
            TUNED.update({k: int(v) for k, v in json.load(f).items()})


load_tuned()


def conv_key(n, hin, win, cin_pad, rows_pad, geom, f32, stats, mask=False):
    """(" mk": the launch also applies a LeakyReLU-backward mask and sums the bias gradient -- another epilogue,
    tuned separately)"""
    return "conv %d %d %d c%d r%d %s%s%s%s" % (n, hin, win, cin_pad, rows_pad, geom.key, " f32" if f32 else "",
                                                " st" if stats else "", " mk" if mask else "")


def wgrad_key(n, ho, wo, cout, cin, r, s, stride):
    return "wgrad %d %d %d co%d ci%d %dx%ds%d" % (n, ho, wo, cout, cin, r, s, stride)


def conv_igemm(x, filt, out, geom, bias=None, act=0, slope=0.0, stats=None, bn_tile=None, k_real=None, n_real=None,
               mask=None, mask_slope=0.0, stats_sum_only=False):
    """out[N,Hout,Wout,rows_pad] = implicit-GEMM conv of x with a packed filter (see pack_filter).
    k_real / n_real: un-padded reduction / output channel counts (for the algorithmic FLOP count).
    mask / mask_slope / stats_sum_only: LeakyReLU backward + bias gradient of the layer that produced
    `mask`, folded into this (data-gradient) launch: out *= leaky'(mask), stats[0] += column sums."""
    n, hin, win, cin, in_ld = _nhwc_meta(x)
    n2, hout, wout, cout_view, out_ld = _nhwc_meta(out)
    rows_pad, n_slabs, cin_pad = filt.shape
    assert n2 == n and hout == geom.Hout and wout == geom.Wout, "output shape mismatch"
    assert cout_view == rows_pad, "output view must expose exactly the packed filter's rows"
    assert x.dtype == torch.bfloat16 and filt.dtype == torch.bfloat16
    out_f32 = 1 if out.dtype == torch.float32 else 0
    if not out_f32:
        assert out.dtype == torch.bfloat16
    if stats is not None:
        assert stats.dtype == torch.float32 and stats.dim() == 2 and stats.shape[0] == 2
    if mask is not None:
        assert mask.dtype == torch.bfloat16 and tuple(mask.shape[:3]) == (n, hout, wout) and mask.shape[3] >= rows_pad
    flops = 2.0 * geom.px_taps * n * (k_real or min(cin, cin_pad)) * (n_real or rows_pad)
    if bn_tile is None:
        key = conv_key(n, hin, win, cin_pad, rows_pad, geom, out_f32, stats is not None and not stats_sum_only, mask is not None)
        bn_tile = TUNED.get(key, 0)
        if RECORD is not None:
            RECORD.append(("conv", key, dict(n=n, hin=hin, win=win, cin=cin, in_ld=in_ld, rows=rows_pad, cin_pad=cin_pad,
                                              n_slabs=n_slabs, geom=geom, f32=out_f32, stats=stats is not None,
                                              bias=bias is not None, out_ld=out_ld, flops=flops, mask=mask is not None,
                                              sum_only=bool(stats_sum_only))))
    call("b200_conv_igemm",
         ptr(x), c_int(in_ld), c_int(0), c_int(cin), c_int(n), c_int(hin), c_int(win),
         ptr(filt), c_int(rows_pad), c_int(cin_pad), c_int(n_slabs),
         ptr(out), c_int(out_ld), c_int(0), c_int(hout), c_int(wout), c_int(out_f32),
         geom.c_n, geom.c_ho, geom.c_wo, geom.c_oa, geom.c_ob, geom.c_nt, geom.c_taps, c_int(geom.tmax),
         c_int(geom.in_stride), c_int(geom.out_stride), ptr(bias), c_int(act), c_float(slope),
         ptr(stats), c_int(0 if stats is None else stats.shape[1]),
         ptr(mask), c_int(0 if mask is None else mask.stride(2)), c_float(mask_slope), c_int(1 if stats_sum_only else 0),
         c_int(bn_tile), stream(), flops=flops,
         tag="M%d N%d K%dx%d s%d/%d%s" % (n * geom.classes[0]["Ho"] * geom.classes[0]["Wo"] * len(geom.classes), rows_pad, cin_pad,
                                            len(geom.classes[0]["taps"]), geom.in_stride, geom.out_stride, " stats" if stats is not None else ""))
    return out


_wgrad_taps = {}


def conv_wgrad(dz, x, dw, r, s, stride, pad, tune=None, scratch=None, taps=None, flops=None, tune_cout=None):
    """dw[Cout,Cin,R,S] (fp32) += sum_pixels dz (x) x ; dz [N,Ho,Wo,>=Cout], x [N,Hin,Win,>=Cin].
    scratch: zeroed fp32 [R*S, Cout, round_up(Cin, 16)] -- accumulate there instead (dw untouched until
    wgrad_unscratch).  taps: explicit [(dh, dw, rs)] list of r*s taps instead of the (r, s, pad) window.
    tune_cout: look the tile up under this output-channel count (the tune word sets the Cin tiling,
    pipeline depth and pixel split only; Cout <= 128 is one row tile whatever its value)."""
    n, ho, wo, _, dz_ld = _nhwc_meta(dz)
    n2, hin, win, _, x_ld = _nhwc_meta(x)
    cout, cin = dw.shape[0], dw.shape[1]
    assert n2 == n and dw.dtype == torch.float32 and dw.is_contiguous()
    tkey = (r, s, pad) if taps is None else tuple(taps)
    taps_c = _wgrad_taps.get(tkey)
    if taps_c is None:
        flat = []
        if taps is None:
            for i in range(r):
                for j in range(s):
                    flat += [i - pad, j - pad, i * s + j]
        else:
            assert len(taps) == r * s
            for t in taps:
                flat += list(t)
        taps_c = _wgrad_taps[tkey] = int_array(flat)
    tap_list, taps = taps, taps_c
    if tune is None:
        key = wgrad_key(n, ho, wo, cout if tune_cout is None else tune_cout, cin, r, s, stride) + ("" if tap_list is None else " v%d" % max(t[1] for t in tap_list))
        tune = TUNED.get(key, 0)
        if RECORD is not None:
            RECORD.append(("wgrad", key, dict(n=n, ho=ho, wo=wo, cout=cout, cin=cin, r=r, s=s, stride=stride, pad=pad,
                                               hin=hin, win=win, dz_c=dz.shape[3], x_c=x.shape[3], dz_ld=dz_ld, x_ld=x_ld,
                                               taps=tap_list, scratch=scratch is not None)))
    call("b200_conv_wgrad",
        ptr(dz), c_int(dz_ld), c_int(0), c_int(cout), c_int(n), c_int(ho), c_int(wo),
        ptr(x), c_int(x_ld), c_int(0), c_int(cin), c_int(hin), c_int(win),
        c_int(r * s), taps, c_int(r * s), c_int(stride), ptr(dw), ptr(scratch),
        c_int(0 if scratch is None else scratch.shape[2]), c_int(tune), stream(),
        flops=flops or 2.0 * n * ho * wo * r * s * cout * cin, tag="px%d co%d ci%d taps%d s%d" % (n * ho * wo, cout, cin, r * s, stride))
    return dw


def wgrad_unscratch_pairview(scratch, dw):
    """dw[Cout, Cin<=32, 4, 4] = pair-view scratch [8, Cout, 64] (see b200_pack_filter in include/b200seg.h)."""
    assert scratch.shape == (8, dw.shape[0], 64) and dw.is_contiguous() and dw.shape[2:] == (4, 4)
    call("b200_wgrad_unscratch_pairview", ptr(scratch), ptr(dw), c_int(dw.shape[0]), c_int(dw.shape[1]), stream(),
         nbytes=8.0 * dw.numel(), tag="pair view")


def wgrad_unscratch(scratch_base, dw_base, table, n_layers, n_weights=0):
    call("b200_wgrad_unscratch", ptr(scratch_base), ptr(dw_base), ptr(table), c_int(n_layers), stream(),
         nbytes=8.0 * n_weights, tag="%d layers" % n_layers)


# ------------------------------------------------------------------ metrics
def fast_hist_accumulate(label, pred, n, hist, bad):
    """hist (int64 [n*n], device) += bincount(n*label+pred) over label in [0,n)."""
    assert label.numel() == pred.numel()
    label = label.contiguous()
    pred = pred.contiguous()
    call("b200_fast_hist", ptr(label), c_int(label.element_size()), ptr(pred),
                               c_int(pred.element_size()), c_int64(label.numel()), c_int(n),
                               ptr(hist), ptr(bad), stream(),
         nbytes=float(label.numel() * (label.element_size() + pred.element_size())), tag="px%d" % label.numel())
    return hist


def count_equal(label, pred, out):
    call("b200_count_equal", ptr(label), c_int(label.element_size()), ptr(pred),
                                 c_int(pred.element_size()), c_int64(label.numel()), ptr(out),
                                 stream(), nbytes=float(label.numel() * (label.element_size() + pred.element_size())),
         tag="px%d" % label.numel())
    return out


def count_equal_batched(label, pred, out):
    """out[i] (int64 [N], device) += #(pred[i] == label[i]) for [N, H, W] maps."""
    n = label.shape[0]
    assert pred.shape == label.shape and out.numel() == n and out.dtype == torch.int64
    label, pred = label.contiguous(), pred.contiguous()
    call("b200_count_equal_batched", ptr(label), c_int(label.element_size()), ptr(pred), c_int(pred.element_size()),
         c_int(n), c_int64(label.numel() // max(n, 1)), ptr(out), stream(),
         nbytes=float(label.numel() * (label.element_size() + pred.element_size())), tag="px%d" % label.numel())
    return out


# ------------------------------------------------------------------ BatchNorm / activation passes
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_SIGMOID = 0, 1, 2, 3


def _pix(t):
    n, h, w, c, ld = _nhwc_meta(t)
    return n * h * w, c, ld


def channel_stats(x, stats):
    npix, c, ld = _pix(x)
    call("b200_channel_stats", ptr(x), c_int(ld), c_int(c), c_int64(npix), ptr(stats), stream(),
         nbytes=2.0 * npix * c, tag="px%d C%d" % (npix, c))


def bn_finalize(stats, count, gamma, beta, running_mean, running_var, training, scale, shift,
                mean, rstd, momentum=0.1, eps=1e-5):
    c = scale.numel()
    call("b200_bn_finalize", ptr(stats), c_int(c), c_float(count), ptr(gamma), ptr(beta),
                                 ptr(running_mean), ptr(running_var), c_float(momentum), c_float(eps),
                                 c_int(1 if training else 0), ptr(scale), ptr(shift), ptr(mean),
                                 ptr(rstd), stream())


def bn_act_apply(x, y, scale, shift, act, slope=0.0):
    npix, c, x_ld = _pix(x)
    npix2, c2, y_ld = _pix(y)
    assert npix == npix2 and c == c2
    call("b200_bn_act_apply", ptr(x), c_int(x_ld), ptr(y), c_int(y_ld), c_int(c), c_int64(npix),
                                  ptr(scale), ptr(shift), c_int(act), c_float(slope), stream(),
         nbytes=4.0 * npix * c, tag="px%d C%d" % (npix, c))


def bn_norm_act(x, y, stats, count, gamma, beta, running_mean, running_var, training, act, slope,
                scale, shift, mean, rstd, momentum=0.1, eps=1e-5):
    npix, c, x_ld = _pix(x)
    call("b200_bn_norm_act", ptr(x), c_int(x_ld), ptr(y), c_int(y.stride(2)), c_int(c), c_int64(npix),
         ptr(stats), c_float(count), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
         c_float(momentum), c_float(eps), c_int(1 if training else 0), c_int(act), c_float(slope),
         ptr(scale), ptr(shift), ptr(mean), ptr(rstd), stream(), nbytes=4.0 * npix * c,
         tag="px%d C%d" % (npix, c))


def bn_act_bwd_reduce(dy1, dy2, z, scale, shift, mean, rstd, act, slope, red):
    npix, c, z_ld = _pix(z)
    call("b200_bn_act_bwd_reduce", 
        ptr(dy1), c_int(dy1.stride(2)), ptr(dy2), c_int(0 if dy2 is None else dy2.stride(2)),
        ptr(z), c_int(z_ld), c_int(c), c_int64(npix), ptr(scale), ptr(shift), ptr(mean), ptr(rstd),
        c_int(act), c_float(slope), ptr(red), stream(),
        nbytes=(4.0 if dy2 is None else 6.0) * npix * c, tag="px%d C%d%s" % (npix, c, "" if dy2 is None else " +dy2"))


def bn_act_bwd_apply(dy1, dy2, z, dz, scale, shift, mean, rstd, red, act, slope):
    npix, c, z_ld = _pix(z)
    call("b200_bn_act_bwd_apply", 
        ptr(dy1), c_int(dy1.stride(2)), ptr(dy2), c_int(0 if dy2 is None else dy2.stride(2)),
        ptr(z), c_int(z_ld), ptr(dz), c_int(dz.stride(2)), c_int(c), c_int64(npix), ptr(scale),
        ptr(shift), ptr(mean), ptr(rstd), ptr(red), c_float(1.0 / npix), c_int(act), c_float(slope),
        stream(), nbytes=(6.0 if dy2 is None else 8.0) * npix * c, tag="px%d C%d%s" % (npix, c, "" if dy2 is None else " +dy2"))


BN_RED_REPLICAS = 8  # kRedRep in csrc/norm.cu


def bn_act_bwd_fused(dy1, dy2, z, dz, scale, shift, mean, rstd, red, act, slope):
    """`red`: zeroed fp32 [1 + BN_RED_REPLICAS, 2, C]; red[0] returns (dbeta, dgamma)."""
    npix, c, z_ld = _pix(z)
    assert red.numel() == (1 + BN_RED_REPLICAS) * 2 * c
    call("b200_bn_act_bwd_fused",
         ptr(dy1), c_int(dy1.stride(2)), ptr(dy2), c_int(0 if dy2 is None else dy2.stride(2)),
         ptr(z), c_int(z_ld), ptr(dz), c_int(dz.stride(2)), c_int(c), c_int64(npix), ptr(scale),
         ptr(shift), ptr(mean), ptr(rstd), ptr(red), c_float(1.0 / npix), c_int(act), c_float(slope),
         stream(), nbytes=(6.0 if dy2 is None else 8.0) * npix * c, tag="px%d C%d%s" % (npix, c, "" if dy2 is None else " +dy2"))


def act_bwd_bias(dy1, dy2, a, dz, act, slope, dbias):
    npix, c, a_ld = _pix(a)
    call("b200_act_bwd_bias", 
        ptr(dy1), c_int(dy1.stride(2)), ptr(dy2), c_int(0 if dy2 is None else dy2.stride(2)),
        ptr(a), c_int(a_ld), ptr(dz), c_int(dz.stride(2)), c_int(c), c_int64(npix), c_int(act),
        c_float(slope), ptr(dbias), stream(), nbytes=(6.0 if dy2 is None else 8.0) * npix * c, tag="px%d C%d" % (npix, c))


# ------------------------------------------------------------------ depthwise / stem
def dwconv_s2_fwd(x, k, w, bias, z, pool, act, slope, stats):
    n, h, wd, c, x_ld = _nhwc_meta(x)
    call("b200_dwconv_s2_fwd", 
        ptr(x), c_int(x_ld), c_int(n), c_int(h), c_int(wd), c_int(c), c_int(k), ptr(w), ptr(bias),
        ptr(z), c_int(z.stride(2)), ptr(pool), c_int(0 if pool is None else pool.stride(2)),
        c_int(act), c_float(slope), ptr(stats), stream(),
        nbytes=2.0 * (x.numel() + z.numel() * (2 if pool is not None else 1)), tag="C%d %dx%d k%d" % (c, h, wd, k))


def dwconv_s2_dgrad(dz, dpool, k, w, dx):
    n, h, wd, c, dx_ld = _nhwc_meta(dx)
    call("b200_dwconv_s2_dgrad", 
        ptr(dz), c_int(dz.stride(2)), ptr(dpool), c_int(0 if dpool is None else dpool.stride(2)),
        c_int(n), c_int(h), c_int(wd), c_int(c), c_int(k), ptr(w), ptr(dx), c_int(dx_ld), stream(),
        nbytes=2.0 * (dx.numel() + dz.numel() * (2 if dpool is not None else 1)), tag="C%d %dx%d k%d" % (c, h, wd, k))


def dwconv_s2_wgrad(dz, x, k, dw, dbias):
    n, h, wd, c, x_ld = _nhwc_meta(x)
    call("b200_dwconv_s2_wgrad", 
        ptr(dz), c_int(dz.stride(2)), ptr(x), c_int(x_ld), c_int(n), c_int(h), c_int(wd), c_int(c),
        c_int(k), ptr(dw), ptr(dbias), stream(), nbytes=2.0 * (x.numel() + dz.numel()), tag="C%d %dx%d k%d" % (c, h, wd, k))


def stem_im2col(img, col):
    """fp32 NCHW image -> bf16 [N, Ho, Wo, 32] unfolded 3x3 stride-2 patches (k = ci*9 + r*3 + s)."""
    n, _, h, wd = img.shape
    assert img.dtype == torch.float32 and img.is_contiguous() and img.shape[1] == 3
    assert col.shape[3] == 32 and col.stride(3) == 1
    call("b200_stem_im2col", ptr(img), c_int(n), c_int(h), c_int(wd), ptr(col), c_int(col.stride(2)), stream(),
         nbytes=4.0 * img.numel() + 2.0 * col.numel(), tag="%dx%d" % (h, wd))
    return col


# ------------------------------------------------------------------ attention
def pool_sum(x, out):
    n, h, w, c, ld = _nhwc_meta(x)
    call("b200_pool_sum", ptr(x), c_int(ld), c_int(n), c_int(h * w), c_int(c), ptr(out), stream(),
         nbytes=2.0 * x.numel(), tag="C%d px%d" % (c, n * h * w))


def fc_small_fwd(inp, in_scale, W, bn, training, act, pre, out, mean, rstd, momentum=0.1, eps=1e-5):
    n, cin = inp.shape
    co = W.shape[0]
    gamma, beta, rm, rv = bn if bn is not None else (None, None, None, None)
    call("b200_fc_small_fwd", 
        ptr(inp), c_float(in_scale), c_int(n), c_int(cin), c_int(co), ptr(W),
        c_int(0 if bn is None else 1), ptr(gamma), ptr(beta), ptr(rm), ptr(rv), c_float(momentum),
        c_float(eps), c_int(1 if training else 0), c_int(act), ptr(pre), ptr(out), ptr(mean), ptr(rstd),
        stream())


def fc_small_bwd(dout, out, pre, inp, in_scale, W, has_bn, training, gamma, mean, rstd, act, scratch,
                 dW, dgamma, dbeta, din, accumulate_din=False):
    n, cin = inp.shape
    co = W.shape[0]
    call("b200_fc_small_bwd", 
        ptr(dout), ptr(out), ptr(pre), ptr(inp), c_float(in_scale), c_int(n), c_int(cin), c_int(co),
        ptr(W), c_int(1 if has_bn else 0), c_int(1 if training else 0), ptr(gamma), ptr(mean), ptr(rstd),
        c_int(act), ptr(scratch), ptr(dW), ptr(dgamma), ptr(dbeta), ptr(din),
        c_int(1 if accumulate_din else 0), stream())


def scale_add_bcast(a, s, s_plus, v, v_scale, t, out):
    n, hs, ws, c, a_ld = _nhwc_meta(a)
    n2, ho, wo, c2, out_ld = _nhwc_meta(out)
    assert n == n2 and c == c2
    call("b200_scale_add_bcast", 
        ptr(a), c_int(a_ld), c_int(hs), c_int(ws), ptr(s), c_float(s_plus), ptr(v), c_float(v_scale),
        ptr(t), c_int(0 if t is None else t.stride(2)), ptr(out), c_int(out_ld), c_int(n), c_int(ho),
        c_int(wo), c_int(c), stream(),
        nbytes=2.0 * (a.numel() + out.numel() + (0 if t is None else t.numel())), tag="C%d %dx%d->%dx%d" % (c, hs, ws, ho, wo))


def upsum_dot_reduce(dout, b, dsum, hs, ws, dot, vsum):
    n, ho, wo, c, dout_ld = _nhwc_meta(dout)
    call("b200_upsum_dot_reduce", 
        ptr(dout), c_int(dout_ld), c_int(ho), c_int(wo), ptr(b), c_int(0 if b is None else b.stride(2)),
        ptr(dsum), c_int(0 if dsum is None else dsum.stride(2)), c_int(n), c_int(hs), c_int(ws),
        c_int(c), ptr(dot), ptr(vsum), stream(),
        nbytes=2.0 * (dout.numel() + (0 if b is None else b.numel()) + (0 if dsum is None else dsum.numel())),
        tag="C%d %dx%d->%dx%d" % (c, ho, wo, hs, ws))


# ------------------------------------------------------------------ up-sampling / losses
UP_LOGITS, UP_CE, UP_SOFTMAX, UP_ARGMAX = 0, 1, 2, 3


def upsample_fwd(lr, H, W, n_classes, mode, out=None, out_flag=0, p_ld=0, labels=None, ignore_index=255,
                 acc=None, loss_map=None):
    n, h_lr, w_lr, ld = lr.shape
    assert lr.dtype == torch.float32 and lr.is_contiguous()
    call("b200_upsample_fwd", 
        ptr(lr), c_int(ld), c_int(n), c_int(h_lr), c_int(w_lr), c_int(H), c_int(W), c_int(n_classes),
        c_int(mode), ptr(out), c_int(out_flag), c_int(p_ld), ptr(labels), c_int(ignore_index), ptr(acc),
        ptr(loss_map), stream(),
        nbytes=float(lr.numel() * 4 + (0 if labels is None else labels.numel() * labels.element_size())
                     + (0 if out is None else n * H * W * (n_classes if out.dim() == 4 and mode != UP_ARGMAX else 1) * out.element_size())
                     + (0 if loss_map is None else loss_map.numel() * 4)),
        tag="mode%d %dx%d" % (mode, H, W))


def upsample_bwd(lr, H, W, n_classes, mode, d_lr, grad_in=None, grad_is_bf16=0, p_ld=0, labels=None,
                 ignore_index=255, pixel_weight=None, coef_num=None, coef_den=None, coef_scale=1.0, loss_acc=None):
    n, h_lr, w_lr, ld = lr.shape
    call("b200_upsample_bwd", 
        ptr(lr), c_int(ld), c_int(n), c_int(h_lr), c_int(w_lr), c_int(H), c_int(W), c_int(n_classes),
        c_int(mode), ptr(grad_in), c_int(grad_is_bf16), c_int(p_ld), ptr(labels), c_int(ignore_index),
        ptr(pixel_weight), ptr(coef_num), ptr(coef_den), c_float(coef_scale), ptr(d_lr), ptr(loss_acc), stream(),
        nbytes=float(lr.numel() * 8 + (0 if labels is None else labels.numel() * labels.element_size())
                     + (0 if grad_in is None else n * H * W * n_classes * grad_in.element_size())
                     + (0 if pixel_weight is None else pixel_weight.numel() * 4)),
        tag="mode%d %dx%d" % (mode, H, W))


# ------------------------------------------------------------------ ADVENT entropy / self-information
ENT_SUM, ENT_MAP = 0, 1            # entropy_fwd: sum of the self-information only / also write the map
ENT_TRAIN, ENT_SELF_INFO = 0, 1    # entropy_bwd: entropy loss + its gradient in one pass / map backward
MAP_PLAIN, MAP_ZERO_BORDERED = 1, 2
ENT_MAP_LD = 32                    # channels per pixel of a self-information map


def check_entropy_args(lr, H, W, n_classes, emap=None, layout=MAP_PLAIN, others=()):
    """The refusals of b200_entropy_fwd / _bwd, raised as ValueError before any device work."""
    if not (isinstance(n_classes, int) and not isinstance(n_classes, bool) and 2 <= n_classes <= 32):
        raise ValueError("n_classes must be an int from 2 to 32, got %r" % (n_classes,))
    if not (isinstance(H, int) and isinstance(W, int) and H >= 1 and W >= 1):
        raise ValueError("H and W must be positive ints, got %r x %r" % (H, W))
    if lr.dim() != 4 or lr.dtype != torch.float32 or not lr.is_contiguous():
        raise ValueError("lr must be contiguous fp32 NHWC [N, h, w, ld], got %s %s" % (lr.dtype, tuple(lr.shape)))
    ld = lr.shape[3]
    if ld % 4 or ld < round_up(n_classes, 4):
        raise ValueError("logits pixel stride %d must be a multiple of 4 and >= %d for %d classes"
                         % (ld, round_up(n_classes, 4), n_classes))
    if emap is not None:
        if layout not in (MAP_PLAIN, MAP_ZERO_BORDERED):
            raise ValueError("map layout %r unknown" % (layout,))
        if layout == MAP_ZERO_BORDERED and (H % 2 or W % 2):
            raise ValueError("the zero-bordered layout needs even H and W, got %d x %d" % (H, W))
        if emap.dim() != 4 or emap.shape[3] != ENT_MAP_LD:
            raise ValueError("map pixel stride must be %d channels, got shape %s" % (ENT_MAP_LD, tuple(emap.shape)))
        hw = (H, W) if layout == MAP_PLAIN else (H + 2, W + 2)
        if emap.dtype != torch.bfloat16 or not emap.is_contiguous() or tuple(emap.shape[:3]) != (lr.shape[0],) + hw:
            raise ValueError("map must be contiguous bf16 %s, got %s %s"
                             % ((lr.shape[0],) + hw + (ENT_MAP_LD,), emap.dtype, tuple(emap.shape)))
    for t in (lr, emap) + tuple(others):
        if t is not None and not t.is_cuda:
            raise ValueError("entropy kernels take CUDA tensors only, got one on %s" % (t.device,))


def entropy_fwd(lr, H, W, n_classes, mode, emap=None, layout=MAP_PLAIN, acc=None):
    """mode ENT_SUM: acc[0] (float64) += sum over pixels and classes of the self-information
    I_c = -p_c log p_c / log n of p = softmax(upsample(lr)); ENT_MAP: also writes I into emap (bf16
    [N, H, W, 32], or [N, H+2, W+2, 32] with a zero border for MAP_ZERO_BORDERED); acc may then be None."""
    if mode not in (ENT_SUM, ENT_MAP) or (mode == ENT_SUM and acc is None) or (mode == ENT_MAP and emap is None):
        raise ValueError("entropy_fwd: mode %r needs %s" % (mode, "acc" if mode == ENT_SUM else "a map"))
    check_entropy_args(lr, H, W, n_classes, emap if mode == ENT_MAP else None, layout, (acc,))
    n, h_lr, w_lr, ld = lr.shape
    call("b200_entropy_fwd", ptr(lr), c_int(ld), c_int(n), c_int(h_lr), c_int(w_lr), c_int(H), c_int(W),
         c_int(n_classes), c_int(mode), ptr(emap if mode == ENT_MAP else None), c_int(ENT_MAP_LD), c_int(layout),
         ptr(acc), stream(),
         nbytes=float(lr.numel() * 4 + (n * H * W * ENT_MAP_LD * 2 if mode == ENT_MAP else 0)),
         tag="mode%d %dx%d" % (mode, H, W))


def entropy_bwd(lr, H, W, n_classes, mode, d_lr, d_map=None, layout=MAP_PLAIN, acc=None):
    """d_lr (fp32, lr's shape) += mode ENT_TRAIN: the gradient of the sum over pixels and classes of I, with
    acc[0] += that sum (acc may be None); ENT_SELF_INFO: the gradient of sum(I * d_map) for the bf16 map
    gradient d_map in the given layout."""
    if mode not in (ENT_TRAIN, ENT_SELF_INFO) or (mode == ENT_SELF_INFO and d_map is None):
        raise ValueError("entropy_bwd: mode %r needs %s" % (mode, "a map gradient" if mode == ENT_SELF_INFO else "d_lr"))
    if d_lr.shape != lr.shape or d_lr.dtype != torch.float32 or not d_lr.is_contiguous():
        raise ValueError("d_lr must be contiguous fp32 of lr's shape %s" % (tuple(lr.shape),))
    check_entropy_args(lr, H, W, n_classes, d_map if mode == ENT_SELF_INFO else None, layout, (d_lr, acc))
    n, h_lr, w_lr, ld = lr.shape
    call("b200_entropy_bwd", ptr(lr), c_int(ld), c_int(n), c_int(h_lr), c_int(w_lr), c_int(H), c_int(W),
         c_int(n_classes), c_int(mode), ptr(d_map if mode == ENT_SELF_INFO else None), c_int(ENT_MAP_LD),
         c_int(layout), ptr(d_lr), ptr(acc if mode == ENT_TRAIN else None), stream(),
         nbytes=float(lr.numel() * 8 + (n * H * W * ENT_MAP_LD * 2 if mode == ENT_SELF_INFO else 0)),
         tag="mode%d %dx%d" % (mode, H, W))


def image_rescale(src, dst, mirror=False):
    """dst = F.interpolate(src, dst.shape[2:], mode='bilinear', align_corners=True) for fp32 NCHW images;
    mirror=True: dst holds 2N images, the second N being torch.flip of the first along the width."""
    n, _, H, W = src.shape
    _, _, h, w = dst.shape
    assert src.dtype == torch.float32 and src.is_contiguous() and dst.dtype == torch.float32 and dst.is_contiguous()
    call("b200_image_rescale", ptr(src), c_int(n), c_int(H), c_int(W), ptr(dst), c_int(h), c_int(w),
         c_int(1 if mirror else 0), stream(), nbytes=4.0 * (src.numel() + dst.numel()), tag="%dx%d->%dx%d" % (H, W, h, w))
    return dst


def msc_argmax(maps, mirrored, H, W, n_classes, pred):
    """pred [N, H, W] (uint8 or int64) = first argmax of the sum over `maps` of softmax(bilinear up-sampling to
    H x W); maps: fp32 NHWC [N, h, w, ld] views (a mirrored half of a 2N forward is ``lr[N:]``), sampled at
    column W-1-x where ``mirrored`` is set."""
    n = pred.shape[0]
    for m in maps:
        assert m.dtype == torch.float32 and m.dim() == 4 and m.is_contiguous() and m.shape[0] == n
    ptrs = (ctypes.c_void_p * len(maps))(*[m.data_ptr() for m in maps])
    call("b200_msc_argmax", c_int(len(maps)), ptrs, int_array([m.shape[3] for m in maps]),
         int_array([m.shape[1] for m in maps]), int_array([m.shape[2] for m in maps]),
         int_array([1 if f else 0 for f in mirrored]), c_int(n), c_int(H), c_int(W), c_int(n_classes), ptr(pred),
         c_int(1 if pred.dtype == torch.uint8 else 0), stream(),
         nbytes=float(sum(m.numel() * 4 for m in maps) + pred.numel() * pred.element_size()),
         tag="%d maps %dx%d" % (len(maps), H, W))
    return pred


def msc_confidence(maps, mirrored, H, W, n_classes, pred, conf):
    """msc_argmax writing pred uint8 [N, H, W] and conf fp32 [N, H, W] = (sum over the maps of the softmax
    probabilities)[pred] / len(maps)."""
    n = pred.shape[0]
    for m in maps:
        assert m.dtype == torch.float32 and m.dim() == 4 and m.is_contiguous() and m.shape[0] == n
    assert pred.dtype == torch.uint8 and conf.dtype == torch.float32 and pred.shape == conf.shape == (n, H, W)
    assert pred.is_contiguous() and conf.is_contiguous()
    ptrs = (ctypes.c_void_p * len(maps))(*[m.data_ptr() for m in maps])
    call("b200_msc_confidence", c_int(len(maps)), ptrs, int_array([m.shape[3] for m in maps]),
         int_array([m.shape[1] for m in maps]), int_array([m.shape[2] for m in maps]),
         int_array([1 if f else 0 for f in mirrored]), c_int(n), c_int(H), c_int(W), c_int(n_classes), ptr(pred),
         ptr(conf), stream(), nbytes=float(sum(m.numel() * 4 for m in maps) + 5 * pred.numel()),
         tag="%d maps %dx%d" % (len(maps), H, W))
    return pred, conf


def class_select_hist(pred, conf, n_classes, pass_, state, hist):
    """One radix pass of the per-class selection over one batch (uint8 pred, fp32 conf, <= 2^30 pixels):
    hist (int64 [n_classes * 256]) += the counts of the next 8 key bits, see include/b200seg.h."""
    assert pred.dtype == torch.uint8 and conf.dtype == torch.float32 and pred.shape == conf.shape
    assert pred.is_contiguous() and conf.is_contiguous()
    assert state.dtype == torch.int64 and hist.dtype == torch.int64
    call("b200_class_select_hist", ptr(pred), ptr(conf), c_int64(pred.numel()), c_int(n_classes), c_int(pass_),
         ptr(state), ptr(hist), stream(), nbytes=5.0 * pred.numel(), tag="pass%d px%d" % (pass_, pred.numel()))


def class_select_pick(n_classes, pass_, portion, cap, state, hist, thr, counts):
    """Fix the next 8 bits of every class's k-th largest key; after pass 3 thr (fp32 [n]) and counts (int64 [n])."""
    assert state.dtype == torch.int64 and hist.dtype == torch.int64
    assert thr.dtype == torch.float32 and counts.dtype == torch.int64
    call("b200_class_select_pick", c_int(n_classes), c_int(pass_), ctypes.c_double(portion), c_float(cap),
         ptr(state), ptr(hist), ptr(thr), ptr(counts), stream())


def pseudo_label_apply(pred, conf, n_classes, thr, out):
    """out = pred where pred < n_classes and conf >= thr[pred], else 255; out uint8 (may be pred) or int64."""
    assert pred.dtype == torch.uint8 and conf.dtype == torch.float32 and pred.shape == conf.shape == out.shape
    assert pred.is_contiguous() and conf.is_contiguous() and out.is_contiguous()
    assert out.dtype in (torch.uint8, torch.int64) and thr.dtype == torch.float32
    call("b200_pseudo_label_apply", ptr(pred), ptr(conf), c_int64(pred.numel()), c_int(n_classes), ptr(thr),
         ptr(out), c_int(1 if out.dtype == torch.uint8 else 0), stream(),
         nbytes=float(pred.numel() * (5 + out.element_size())), tag="px%d" % pred.numel())
    return out


def radix_select_desc(x, rank, state, hist):
    call("b200_radix_select_desc", ptr(x), c_int64(x.numel()), c_int64(rank), ptr(state), ptr(hist),
                                       stream(), nbytes=16.0 * x.numel(), tag="n%d" % x.numel())


def ohem_reduce(x, state, threshold, keep_num, sums, out):
    call("b200_ohem_reduce", ptr(x), c_int64(x.numel()), ptr(state), c_float(threshold),
                                 c_int64(keep_num), ptr(sums), ptr(out), stream(), nbytes=4.0 * x.numel(), tag="n%d" % x.numel())


def ohem_weights(x, sel, wout):
    call("b200_ohem_weights", ptr(x), c_int64(x.numel()), ptr(sel), ptr(wout), stream(), nbytes=8.0 * x.numel(),
         tag="n%d" % x.numel())


def bce_const_fwd(x, target, out):
    call("b200_bce_const_fwd", ptr(x), c_int(x.numel()), c_float(target), ptr(out), stream())


def bce_const_bwd(x, target, gscale, gmul, dx):
    call("b200_bce_const_bwd", ptr(x), c_int(x.numel()), c_float(target), ptr(gscale), c_float(gmul),
                                   ptr(dx), stream())


# ------------------------------------------------------------------ discriminator classifier
def classifier_fwd(x, w, bias, out):
    n, h, wd, c, ld = _nhwc_meta(x)
    call("b200_classifier_fwd", ptr(x), c_int(ld), c_int(n), c_int(h), c_int(wd), c_int(c), ptr(w),
                                    ptr(bias), ptr(out), stream(), nbytes=2.0 * x.numel(), tag="C%d %dx%d" % (c, h, wd))


def classifier_dgrad(dout, w, dx):
    n, h, wd, c, ld = _nhwc_meta(dx)
    call("b200_classifier_dgrad", ptr(dout), c_int(n), c_int(h), c_int(wd), c_int(c), ptr(w), ptr(dx),
                                      c_int(ld), stream(), nbytes=2.0 * dx.numel(), tag="C%d %dx%d" % (c, h, wd))


def classifier_wgrad(dout, x, dw, dbias):
    n, h, wd, c, ld = _nhwc_meta(x)
    call("b200_classifier_wgrad", ptr(dout), ptr(x), c_int(ld), c_int(n), c_int(h), c_int(wd), c_int(c),
                                      ptr(dw), ptr(dbias), stream(), nbytes=2.0 * x.numel(), tag="C%d %dx%d" % (c, h, wd))


def cast_f32_bf16(x, y):
    assert x.is_contiguous() and y.is_contiguous() and x.numel() == y.numel()
    call("b200_cast_f32_bf16", ptr(x), ptr(y), c_int64(x.numel()), stream(), nbytes=6.0 * x.numel(), tag="n%d" % x.numel())
    return y


def scale_f32(x, num, den, mul, y):
    call("b200_scale_f32", ptr(x), c_int64(x.numel()), ptr(num), ptr(den), c_float(mul), ptr(y), stream(),
         nbytes=8.0 * x.numel(), tag="n%d" % x.numel())
    return y


# ------------------------------------------------------------------ input pipeline
def image_resize_normalize(src, xb, xk, yb, yk, lut, dst, max_rows):
    """uint8 [N, H0, W0, 3] -> fp32 [N, 3, H, W]: Pillow's two-pass bilinear resample + the
    ToTensor/Normalize table (dataset/cityscapes.py:65,67).  Tables come from ``dataset.ResizeTables``."""
    n, h0, w0, c = src.shape
    assert c == 3 and src.dtype == torch.uint8 and src.is_contiguous()
    _, _, h, w = dst.shape
    assert dst.dtype == torch.float32 and dst.is_contiguous() and dst.shape[1] == 3
    call("b200_image_resize_normalize", ptr(src), c_int(n), c_int(h0), c_int(w0), ptr(xb), ptr(xk),
         c_int(xk.shape[1]), ptr(yb), ptr(yk), c_int(yk.shape[1]), c_int(h), c_int(w), ptr(lut), ptr(dst),
         c_int(max_rows), stream(), nbytes=float(src.numel() + 4 * dst.numel()), tag="%dx%d->%dx%d" % (h0, w0, h, w))
    return dst


def label_resize_remap(src, ix, iy, lut, dst):
    """uint8 [N, H0, W0] -> uint8 / int64 [N, H, W]: Pillow's NEAREST resize + a 256-entry id remap."""
    n, h0, w0 = src.shape
    assert src.dtype == torch.uint8 and src.is_contiguous() and dst.is_contiguous()
    h, w = dst.shape[-2:]
    assert dst.dtype in (torch.uint8, torch.int64)
    call("b200_label_resize_remap", ptr(src), c_int(n), c_int(h0), c_int(w0), ptr(ix), ptr(iy), c_int(h),
         c_int(w), ptr(lut), ptr(dst), c_int(1 if dst.dtype == torch.int64 else 0), stream(),
         nbytes=float(src.numel() + dst.numel() * dst.element_size()), tag="%dx%d->%dx%d" % (h0, w0, h, w))
    return dst
