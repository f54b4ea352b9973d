"""Layer-level forward/backward built from the CUDA kernels (no autograd in here).

Each ``*_fwd`` returns ``(output, ctx)`` and each ``*_bwd`` consumes that ctx.  Activations are
bf16 NHWC tensors ``[N, H, W, C]`` (channel slices of wider buffers are fine, see kernels.py);
parameters stay the fp32 ``nn.Parameter`` masters, their bf16 GEMM packings are cached per
parameter version.  torch is used for allocation only.
"""
import torch

from . import kernels as K

BF16 = torch.bfloat16
F32 = torch.float32

# debugging aid: when True every filter is re-packed on every use (the normal policy is in
# refresh_packs: always in training mode and after any backward, otherwise on version change)
FORCE_REPACK = False


def packed_filter(weight, transpose, shape=None, rows_pad=None):
    """bf16 GEMM packing of a conv filter, cached ON the parameter object (so it dies with it and a
    recycled device address can never alias a stale packing) and refreshed when the parameter's
    version counter or storage changes (optimizer steps, load_state_dict, .to()).  ``shape``
    reinterprets the filter memory (the stem's [32, 3, 3, 3] as a [32, 27, 1, 1] 1x1 filter);
    ``rows_pad`` widens the packed rows beyond the multiple of 16 (zero rows)."""
    cache = getattr(weight, "_b200_pack", None)
    if cache is None:
        cache = {}
        try:
            weight._b200_pack = cache
        except AttributeError:
            pass
    shape = tuple(shape) if shape is not None else tuple(weight.shape)
    key = (int(transpose), shape)
    ver, ptr_now = weight._version, weight.data_ptr()
    hit = cache.get(key)
    if hit is not None and hit[0] == ver and hit[1] == ptr_now and not FORCE_REPACK:
        return hit[2]
    w = weight.detach().view(shape)
    if hit is not None and hit[2].device == weight.device:
        buf = hit[2]  # repack in place: stable pointer for graphs, no allocator churn
        cout, cin, r, s = shape
        K.call("b200_pack_filter", K.ptr(w), K.ptr(buf), K.c_int(cout), K.c_int(cin), K.c_int(r * s),
               K.c_int(buf.shape[0]), K.c_int(buf.shape[2]), K.c_int(int(transpose)), K.stream())
    else:
        buf = K.pack_filter(w, transpose, rows_pad)
    cache[key] = (ver, ptr_now, buf)
    return buf


def packed_filter_pairview(weight, transpose):
    """Pair-view packing [64][8][64] of a 4x4 / stride-2 / pad-1 filter with <= 32 input channels (the dense
    discriminator's first layer over the zero-bordered probability map, see include/b200seg.h
    b200_pack_filter); cached and batch-refreshed like every other packing (mode 2 / 3 of the pack kernels)."""
    cout, cin, r, s = weight.shape
    assert (r, s) == (4, 4) and cin <= 32 and cout % 16 == 0
    mode = 3 if transpose else 2
    cache = getattr(weight, "_b200_pack", None)
    if cache is None:
        cache = {}
        weight._b200_pack = cache
    key = (mode, (cout, cin, 8, 1))
    ver, ptr_now = weight._version, weight.data_ptr()
    hit = cache.get(key)
    if hit is not None and hit[0] == ver and hit[1] == ptr_now and not FORCE_REPACK:
        return hit[2]
    if hit is not None and hit[2].device == weight.device:
        buf = hit[2]
    else:
        buf = torch.empty((64, 8, cout) if transpose else (cout, 8, 64), dtype=BF16, device=weight.device)
    K.call("b200_pack_filter", K.ptr(weight.detach()), K.ptr(buf), K.c_int(cout), K.c_int(cin), K.c_int(8),
           K.c_int(buf.shape[0]), K.c_int(buf.shape[2]), K.c_int(mode), K.stream())
    cache[key] = (ver, ptr_now, buf)
    return buf


def refresh_packs(module, force=False):
    """Re-pack, in ONE launch, every cached filter packing of `module` whose fp32 master changed
    (called at the top of a forward; after an optimizer step that is all of them).

    Staleness cannot rely on tensor version counters alone: torch's fused optimizers update
    parameters without bumping them.  So `force` is set by the caller whenever the weights may have
    been stepped since the last packing: always in training mode, and after any backward pass
    through the module (see _glue.run_module).  Out-of-band edits through ``.data`` need
    ``invalidate_packs(module)``."""
    weights = getattr(module, "_b200_conv_weights", None)
    if weights is None:
        weights = [p for p in module.parameters() if p.dim() == 4]
        object.__setattr__(module, "_b200_conv_weights", weights)
    stale = []
    for w in weights:
        cache = getattr(w, "_b200_pack", None)
        if not cache:
            continue
        ver, ptr_now = w._version, w.data_ptr()
        for key, (v, pw, buf) in cache.items():
            if v != ver or pw != ptr_now or FORCE_REPACK or force:
                stale.append((w, key, buf))
    if not stale:
        return 0
    key = tuple((w.data_ptr(), k, buf.data_ptr()) for w, k, buf in stale)
    tab = getattr(module, "_b200_pack_table", None)
    if tab is None or tab[0] != key:
        rows = []
        for w, (tr, shape), buf in stale:
            cout, cin, r, s = shape
            rows.append([w.data_ptr(), buf.data_ptr(), cout, cin, r * s, buf.shape[0], buf.shape[2], int(tr)])
        dev = torch.tensor(rows, dtype=torch.int64).to(stale[0][0].device)
        nbytes = float(sum(4 * w.numel() + 2 * buf.numel() for w, _, buf in stale))
        tab = (key, dev, nbytes)
        object.__setattr__(module, "_b200_pack_table", tab)
    K.call("b200_pack_filters_batched", K.ptr(tab[1]), K.c_int(len(stale)), K.stream(), nbytes=tab[2],
           tag="%d filters" % len(stale))
    for w, k, buf in stale:
        w._b200_pack[k] = (w._version, w.data_ptr(), buf)
    return len(stale)


def invalidate_packs(module):
    """Force the next forward of `module` to re-pack every filter (after editing weights in place)."""
    object.__setattr__(module, "_b200_dirty", True)


class _ZeroArena(object):
    """fp32 zero-initialised scratch carved out of ONE torch.zeros per module forward / backward
    (instead of one memset launch per BatchNorm statistic, gradient accumulator, ...).  Every
    begin() starts a fresh allocation, so tensors handed out earlier (e.g. parameter gradients kept
    by autograd) are never recycled; the size needed per (module, phase) is remembered."""

    def __init__(self):
        self.hint = {}
        self.stack = []

    def begin(self, tag, device):
        self.stack.append([tag, device, None, 0, 0, 0])  # tag, device, chunk, offset, requested, all-reduced mark

    def end(self):
        tag, _, _, _, requested, _ = self.stack.pop()
        self.hint[tag] = max(self.hint.get(tag, 0), requested)

    def zeros(self, shape, device):
        n = 1
        for d in shape:
            n *= int(d)
        if not self.stack or self.stack[-1][1] != device:
            return torch.zeros(shape, dtype=F32, device=device)
        st = self.stack[-1]
        size = (n + 63) // 64 * 64
        st[4] += size
        if st[2] is None or st[3] + size > st[2].numel():
            st[2] = torch.zeros(max(size, self.hint.get(st[0], 0) - (st[4] - size), 1 << 16), dtype=F32, device=device)
            st[3] = 0
            st[5] = 0   # (an un-reduced tail of the retired chunk is picked up by the flat fallback)
        out = st[2][st[3]:st[3] + n].view(shape)
        st[3] += size
        return out


ARENA = _ZeroArena()


class _GradReducer(object):
    """Data-parallel gradient exchange overlapped with the backward, with no flatten / unflatten copies.

    Every parameter gradient of a module backward is a slice of the arena chunk above, handed out in
    the order the backward produces them.  So "the gradients finished so far" is one contiguous fp32
    span: `hook()` (called by the model backwards after their parameter-heavy late stages, and once
    at the end) all-reduces the span produced since the previous hook IN PLACE on a communication
    stream while the main stream keeps running the rest of the backward.  The span also contains
    consumed scratch (BatchNorm partial sums); averaging that is harmless.  `finish()` makes the
    main stream wait for the exchange and returns the gradients that were not covered (first
    iterations, before the arena knows its size; gradients made by other autograd nodes)."""

    MIN_FLOATS = 1 << 20

    def __init__(self):
        self.active = False
        self.streams = {}
        self.spans = []
        self.snapshots = None   # tests: list that receives (span view, copy of the span before the exchange)
        self.force = False      # tests: take the overlapped path on a 1-rank NCCL group too
        self.dropped = 0        # backwards that found accumulated gradients and fell back to the flat exchange

    @staticmethod
    def world():
        import torch.distributed as dist
        return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1

    def begin(self, need_dw, device, params=()):
        """Called at the top of a module backward.  `params`: the module's parameters.

        The in-place exchange is only valid for the FIRST backward after zero_grad(): autograd then
        adopts the arena slice as ``p.grad``.  When a parameter already holds a gradient
        (train_da_step_nni accumulates two backwards per optimizer step, train_nni.py:118-139),
        autograd will run ``p.grad += new`` on the main stream -- so this backward is not exchanged
        span by span, the main stream first waits for any exchange still in flight on ``p.grad``, and
        the spans that hold such gradients are forgotten: ``finish()`` then hands those gradients to
        the flat all-reduce (averaging an already averaged part again is the identity on it)."""
        import torch.distributed as dist
        self.active = bool(need_dw) and device.type == "cuda" and (self.world() > 1 or self.force) and \
            dist.is_initialized() and dist.get_backend() == "nccl"
        if not self.active:
            return
        held = [p.grad for p in params if p.grad is not None]
        if held:
            self.active = False
            if self.spans:
                for key, comm in self.streams.items():
                    torch.cuda.current_stream(torch.device("cuda", key)).wait_stream(comm)
                ptrs = [g.data_ptr() for g in held]
                self.spans = [sp for sp in self.spans if not any(sp[0] <= q < sp[1] for q in ptrs)]
                self.dropped += 1

    def hook(self, final=False):
        if not self.active or not ARENA.stack:
            return
        st = ARENA.stack[-1]
        chunk, lo, hi = st[2], st[5], st[3]
        if chunk is None or hi - lo < (1 if final else self.MIN_FLOATS):
            return
        import torch.distributed as dist
        dev = st[1]
        key = dev.index or 0
        if key not in self.streams:
            self.streams[key] = torch.cuda.Stream(device=dev)
        comm, main = self.streams[key], torch.cuda.current_stream(dev)
        WSCRATCH.flush()   # gradients accumulated in tap-major scratch become final first
        view = chunk[lo:hi]
        comm.wait_stream(main)
        with torch.cuda.stream(comm):
            if self.snapshots is not None:
                self.snapshots.append((view, view.clone()))
            dist.all_reduce(view, op=dist.ReduceOp.AVG)
        self.spans.append((view.data_ptr(), view.data_ptr() + 4 * view.numel(), view))
        st[5] = hi

    def end(self):
        self.hook(final=True)
        self.active = False

    def finish(self, grads):
        """-> the gradients still to be exchanged; the main stream now waits for the spans."""
        if not self.spans:
            return grads
        for key, comm in self.streams.items():
            torch.cuda.current_stream(torch.device("cuda", key)).wait_stream(comm)
        left = []
        for g in grads:
            ptr = g.data_ptr()
            if not (g.dtype == F32 and any(lo <= ptr and ptr + 4 * g.numel() <= hi for lo, hi, _ in self.spans)):
                left.append(g)
        self.spans = []
        return left


REDUCER = _GradReducer()


def zeros_f32(shape, device):
    return ARENA.zeros(tuple(shape) if not isinstance(shape, int) else (shape,), device)


def empty_act(n, h, w, c, device):
    return torch.empty((n, h, w, c), dtype=BF16, device=device)


# --------------------------------------------------------------------------- BatchNorm (+act)
class BNCtx:
    __slots__ = ("z", "scale", "shift", "mean", "rstd", "act", "slope", "training")


def bn_act_fwd(z, stats, bn, training, act, slope=0.0, out=None):
    """z: raw conv output; stats: [2, C] sums (train) or None (eval); bn = (gamma, beta, rm, rv)."""
    n, h, w, c = z.shape
    gamma, beta, rm, rv = bn
    buf = torch.empty((4, c), dtype=F32, device=z.device)
    a = out if out is not None else torch.empty_like(z)
    K.bn_norm_act(z, a, stats, float(n * h * w), gamma, beta, rm, rv, training, act, slope,
                  buf[0], buf[1], buf[2], buf[3])
    ctx = BNCtx()
    ctx.z, ctx.scale, ctx.shift, ctx.mean, ctx.rstd = z, buf[0], buf[1], buf[2], buf[3]
    ctx.act, ctx.slope, ctx.training = act, slope, training
    return a, ctx


def bn_act_bwd(ctx, dy1, dy2=None):
    """-> (dz, dgamma, dbeta) for train-mode BatchNorm followed by ctx.act."""
    if not ctx.training:
        raise NotImplementedError("backward through eval-mode BatchNorm is not part of the reference's training path")
    c = ctx.z.shape[3]
    red = zeros_f32((1 + K.BN_RED_REPLICAS, 2, c), ctx.z.device)   # [0]: totals, [1:]: partial-sum replicas
    dz = torch.empty(ctx.z.shape, dtype=BF16, device=ctx.z.device)
    K.bn_act_bwd_fused(dy1, dy2, ctx.z, dz, ctx.scale, ctx.shift, ctx.mean, ctx.rstd, red, ctx.act, ctx.slope)
    return dz, red[0, 1], red[0, 0]


# --------------------------------------------------------------------------- dense conv (+BN+act)
class ConvCtx:
    __slots__ = ("x", "weight", "stride", "pad", "bn", "a", "act", "slope", "stem_col")


def conv_raw_fwd(x, weight, stride, pad, stats=None, bias=None, act=K.ACT_NONE, slope=0.0, out=None,
                 out_dtype=BF16, rows_pad=None):
    """Implicit-GEMM convolution of an NHWC bf16 view; returns the [N,Ho,Wo,rows_pad] result."""
    n, h, w, _ = x.shape
    _, _, r, s = weight.shape
    geom = K.fwd_geometry(h, w, r, s, stride, pad)
    filt = packed_filter(weight, False, rows_pad=rows_pad)
    if out is None:
        out = torch.empty((n, geom.Hout, geom.Wout, filt.shape[0]), dtype=out_dtype, device=x.device)
    K.conv_igemm(x, filt, out, geom, bias=bias, act=act, slope=slope, stats=stats,
                 k_real=weight.shape[1], n_real=weight.shape[0])
    return out


def conv_dgrad(dz, weight, stride, pad, hin, win, mask=None, mask_slope=0.0, dbias=None):
    """dx[N,hin,win,round16(Cin)] of a dense conv given dz (NHWC bf16 view over the conv's output).
    With `mask` (the stored activation of the layer that produced this conv's input) the launch also
    applies that layer's LeakyReLU backward, i.e. it returns the producer's dz directly, and
    accumulates the producer's bias gradient into dbias[0] (fp32 [2, round16(Cin)], zeroed)."""
    _, _, r, s = weight.shape
    geom = K.dgrad_geometry(hin, win, r, s, stride, pad)
    filt_t = packed_filter(weight, True)
    dx = torch.empty((dz.shape[0], hin, win, filt_t.shape[0]), dtype=BF16, device=dz.device)
    K.conv_igemm(dz, filt_t, dx, geom, k_real=weight.shape[0], n_real=weight.shape[1], mask=mask,
                 mask_slope=mask_slope, stats=dbias, stats_sum_only=dbias is not None)
    return dx


class _WgradScratch(object):
    """Tap-major scratch accumulators of the multi-tap weight gradients of ONE module backward.

    The split-K partials of a 3x3 / 4x4 layer land in dW[co][ci][rs] 4*RS bytes apart: 16 scalar
    atomics per thread and chunk (0.8 ms of a 15.3 ms step).  Inside a module backward they are
    accumulated instead into scratch[rs][co][ci] (16-byte vector reductions) carved from a second
    zero arena, and ONE launch at the end of the backward permutes every layer into its dW.  That
    launch addresses the layers by their offsets inside the two arena chunks -- stable once the
    arenas know their size (from the fourth eager step of a kind on) -- so its table is uploaded
    during the eager warm-up and never inside a CUDA-graph capture (a capture taken earlier simply
    keeps the scalar-atomic path)."""

    def __init__(self):
        self.arena = _ZeroArena()
        self.depth = 0
        self.pending = []
        self.tables = {}
        self.tag = None
        self.seen = {}        # tag -> the row sets flushed during the previous backward of that kind
        self.stable = {}      # tag -> the last two backwards of that kind flushed identical row sets
        self.flushed = []

    def begin(self, tag, device):
        self.arena.begin(tag, device)
        self.depth += 1
        self.pending, self.flushed, self.tag = [], [], tag

    def request(self, dw, cout, cin, rs):
        """-> scratch tensor or None (not inside a module backward / arenas not settled / thin layer)."""
        if self.depth == 0 or rs == 1 or cin <= 32 or not ARENA.stack:
            return None
        dchunk = ARENA.stack[-1][2]
        if dchunk is None or self.arena.hint.get(self.tag) is None:
            return None
        if torch.cuda.is_current_stream_capturing() and not self.stable.get(self.tag):
            return None          # layout not settled yet (needs 4 eager steps): no table upload inside a capture
        ci_pad = (cin + 15) // 16 * 16
        sc = self.arena.zeros((rs, cout, ci_pad), dw.device)
        schunk = self.arena.stack[-1][2]
        d_off = (dw.data_ptr() - dchunk.data_ptr()) // 4
        s_off = (sc.data_ptr() - schunk.data_ptr()) // 4
        if not (0 <= d_off and d_off + dw.numel() <= dchunk.numel() and 0 <= s_off and s_off + sc.numel() <= schunk.numel()):
            return None
        if self.pending and (self.pending[0][0] is not schunk or self.pending[0][1] is not dchunk):
            self.flush()         # an arena grew mid-backward: close the batch of the old chunks
        self.pending.append((schunk, dchunk, (s_off, d_off, cout, cin, rs, ci_pad)))
        return sc

    def flush(self):
        """Permute the scratch accumulators gathered so far into their gradients (one launch).  Also
        called by REDUCER.hook(): a gradient span must be final before it is exchanged."""
        SIDE.join()    # weight gradients still running on the side stream
        if not self.pending:
            return
        schunk, dchunk = self.pending[0][0], self.pending[0][1]
        rows = tuple(p[2] for p in self.pending)
        tab = self.tables.get(rows)
        if tab is None:
            if torch.cuda.is_current_stream_capturing():
                raise K._lib.B200Error("weight-gradient scratch layout changed inside a CUDA-graph capture: "
                                       "run the step eagerly (three times) before capturing")
            tab = self.tables[rows] = torch.tensor(rows, dtype=torch.int64).to(schunk.device)
        K.wgrad_unscratch(schunk, dchunk, tab, len(rows), sum(r_[2] * r_[3] * r_[4] for r_ in rows))
        self.flushed.append(rows)
        self.pending = []

    def end(self, ok=True):
        SIDE.join()
        if ok:
            self.flush()
            self.stable[self.tag] = bool(self.flushed) and self.flushed == self.seen.get(self.tag)
            self.seen[self.tag] = self.flushed
        self.pending = []
        self.depth -= 1
        self.arena.end()


WSCRATCH = _WgradScratch()


class _SideStream(object):
    """Weight gradients of SMALL layers run on a second stream, concurrently with the data gradient of the
    same layer (both only read dz; nothing reads dW before the end of the module backward).  At 1/16 and 1/32
    resolution either kernel is a few dozen CTAs with a 10-20 us latency chain, so the pair fits the GPU side
    by side; large layers fill every SM on their own and stay in line (overlap bought nothing there).
    Inside a CUDA-graph capture the fork / join become graph edges.  Tensors the side kernels touch are
    kept alive until the join (the caching allocator would hand a freed block to the main stream at once)."""

    def __init__(self):
        self.streams = {}
        self.keep = []
        self.dirty = None

    def run(self, device, keep, fn):
        key = device.index or 0
        side = self.streams.get(key)
        if side is None:
            side = self.streams[key] = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            fn()
        self.keep.append(keep)
        self.dirty = (device, side)

    def join(self):
        if self.dirty is not None:
            device, side = self.dirty
            torch.cuda.current_stream(device).wait_stream(side)
            self.dirty = None
            self.keep = []


SIDE = _SideStream()
# layers with at most this many output pixels (N*Ho*Wo) send their weight gradient to the side stream (0 = off).
# Measured on the DA step (N = 8, 512x1024, graph replay): 0 -> 11.89 ms, 16384 -> 11.83, 65536 -> 11.70,
# 262144 and beyond -> 11.68-11.71 (the large layers fill the GPU alone: nothing more to overlap).
WGRAD_SIDE_MAX_PIXELS = 65536


def conv_wgrad(dz, x, weight, stride, pad, tune_cout=None):
    cout, cin, r, s = weight.shape
    dw = zeros_f32((cout, cin, r, s), dz.device)
    scratch = WSCRATCH.request(dw, cout, cin, r * s)
    if WSCRATCH.depth > 0 and dz.shape[0] * dz.shape[1] * dz.shape[2] <= WGRAD_SIDE_MAX_PIXELS:
        SIDE.run(dz.device, (dz, x, dw, scratch),
                 lambda: K.conv_wgrad(dz, x, dw, r, s, stride, pad, scratch=scratch, tune_cout=tune_cout))
    else:
        K.conv_wgrad(dz, x, dw, r, s, stride, pad, scratch=scratch, tune_cout=tune_cout)
    return dw


def conv_bn_act_fwd(x, weight, bn, stride, pad, training, act=K.ACT_RELU, slope=0.0, out=None):
    """ConvX / ConvBNReLU: bias-free conv -> BatchNorm2d -> activation (stdcnet.py:6-15,
    model_stages.py:11-29).  `x` is an NHWC bf16 view, or the fp32 NCHW image for the 3-channel stem."""
    cout = weight.shape[0]
    stats = zeros_f32((2, cout), weight.device) if training else None
    ctx = ConvCtx()
    ctx.stem_col = None
    if x.dim() == 4 and x.dtype == F32 and x.shape[1] == 3 and weight.shape[1] == 3:
        # stem: unfold the NCHW image once (bf16, 32 values per output pixel), then a K = 32 1x1 GEMM
        assert weight.shape[2] == 3 and stride == 2 and pad == 1 and cout == 32
        n, _, h, w = x.shape
        ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
        col = K.stem_im2col(x, empty_act(n, ho, wo, 32, x.device))
        z = empty_act(n, ho, wo, cout, x.device)
        K.conv_igemm(col, packed_filter(weight, False, (cout, 27, 1, 1)), z, K.fwd_geometry(ho, wo, 1, 1, 1, 0),
                     stats=stats, k_real=27, n_real=cout)
        ctx.stem_col = col
    else:
        assert cout % 16 == 0, "BatchNorm'd convs have a multiple of 16 output channels"
        z = conv_raw_fwd(x, weight, stride, pad, stats=stats)
    a, bnctx = bn_act_fwd(z, stats, bn, training, act, slope, out)
    ctx.x, ctx.weight, ctx.stride, ctx.pad, ctx.bn, ctx.a = x, weight, stride, pad, bnctx, a
    ctx.act, ctx.slope = act, slope
    return a, ctx


def conv_bn_act_bwd(ctx, dy1, dy2=None, need_dx=True):
    """-> (dx or None, dW, dgamma, dbeta)"""
    dz, dgamma, dbeta = bn_act_bwd(ctx.bn, dy1, dy2)
    if ctx.stem_col is not None:
        dw = zeros_f32(ctx.weight.shape, dz.device)
        K.conv_wgrad(dz, ctx.stem_col[..., :27], dw.view(dw.shape[0], 27, 1, 1), 1, 1, 1, 0)
        return None, dw, dgamma, dbeta
    dw = conv_wgrad(dz, ctx.x, ctx.weight, ctx.stride, ctx.pad)
    dx = None
    if need_dx:
        dx = conv_dgrad(dz, ctx.weight, ctx.stride, ctx.pad, ctx.x.shape[1], ctx.x.shape[2])
    return dx, dw, dgamma, dbeta


# --------------------------------------------------------------------------- biased conv + LeakyReLU
class ConvBiasCtx:
    __slots__ = ("x", "weight", "stride", "pad", "a", "act", "slope", "has_bias", "pairview")


def conv_pairview_fwd(xpad, weight, bias_padded, act, slope):
    """FCDiscriminator.conv1 (discriminator.py:9,18: Conv2d(C<=32, ndf, 4, 2, 1) + LeakyReLU) over the
    zero-bordered probability buffer xpad [N, H+2, W+2, 32]: a stride-1 filter of 8 taps over its column-pair
    view [N, (H+2)/2, W+2, 64] (kernels.pairview_fwd_geometry) -- 128-byte stride-1 TMA rows and K = 8 x 64
    instead of 16 taps of 64-byte stride-2 rows."""
    n, hp, wp, c = xpad.shape
    assert c == 32 and xpad.is_contiguous() and hp % 2 == 0 and wp % 2 == 0
    h, w = hp - 2, wp - 2
    cout, cin = weight.shape[0], weight.shape[1]
    xv = xpad.view(n, hp // 2, wp, 64)
    a = torch.empty((n, h // 2, w // 2, cout), dtype=BF16, device=xpad.device)
    K.conv_igemm(xv, packed_filter_pairview(weight, False), a, K.pairview_fwd_geometry(h, w), bias=bias_padded, act=act,
                 slope=slope, k_real=2 * cin, n_real=cout)
    ctx = ConvBiasCtx()
    ctx.x, ctx.weight, ctx.stride, ctx.pad, ctx.a, ctx.act, ctx.slope = xv, weight, 2, 1, a, act, slope
    ctx.pairview = (h, w)
    return a, ctx


def _pairview_wgrad(ctx, dz):
    h, w = ctx.pairview
    cout, cin = ctx.weight.shape[0], ctx.weight.shape[1]
    sc = zeros_f32((8, cout, 64), dz.device)
    taps = K.pairview_fwd_geometry(h, w).classes[0]["taps"]
    K.conv_wgrad(dz, ctx.x, sc.view(cout, 64, 8, 1), 8, 1, 1, 0, scratch=sc, taps=taps,
                 flops=2.0 * dz.shape[0] * dz.shape[1] * dz.shape[2] * 16 * cout * cin)
    dw = zeros_f32(ctx.weight.shape, dz.device)
    K.wgrad_unscratch_pairview(sc, dw)
    return dw


def _pairview_dgrad(ctx, dz):
    """-> d(probabilities) as the interior view [N, H, W, 32] of a [N, H+2, W+2, 32] buffer (border = junk)."""
    h, w = ctx.pairview
    cout, cin = ctx.weight.shape[0], ctx.weight.shape[1]
    n = dz.shape[0]
    dxv = torch.empty((n, (h + 2) // 2, w + 2, 64), dtype=BF16, device=dz.device)
    K.conv_igemm(dz, packed_filter_pairview(ctx.weight, True), dxv, K.pairview_dgrad_geometry(h, w), k_real=cout,
                 n_real=2 * cin)
    return dxv.view(n, h + 2, w + 2, 32)[:, 1:h + 1, 1:w + 1]


def conv_bias_act_fwd(x, weight, bias_padded, stride, pad, act, slope):
    """FCDiscriminator layers (discriminator.py:17-25): conv + bias + LeakyReLU fused in the epilogue."""
    a = conv_raw_fwd(x, weight, stride, pad, bias=bias_padded, act=act, slope=slope)
    ctx = ConvBiasCtx()
    ctx.x, ctx.weight, ctx.stride, ctx.pad, ctx.a, ctx.act, ctx.slope = x, weight, stride, pad, a, act, slope
    ctx.pairview = None
    return a, ctx


def conv_bias_act_bwd(ctx, dy1, dy2=None, need_dx=True, need_dw=True, dz_dbias=None, producer=None):
    """-> (dx, dW, dbias).

    dz_dbias = (dz, dbias): this layer's activation backward was already folded into the launch
    that produced its output gradient (see `producer`), dy1 is ignored.
    producer = ConvCtx of the biased conv + LeakyReLU layer that produced this layer's input: its
    activation backward and bias gradient are folded into this layer's data-gradient launch and
    `dx` is returned as the pair (producer's dz, producer's dbias) for the next call."""
    c = ctx.a.shape[3]
    if dz_dbias is not None:
        dz, dbias = dz_dbias
    else:
        dz = torch.empty(ctx.a.shape, dtype=BF16, device=ctx.a.device)
        dbias = zeros_f32((c,), ctx.a.device) if need_dw else None
        K.act_bwd_bias(dy1, dy2, ctx.a, dz, ctx.act, ctx.slope, dbias)
    if ctx.pairview is not None:
        dw = _pairview_wgrad(ctx, dz) if need_dw else None
        dx = _pairview_dgrad(ctx, dz) if need_dx else None
        if dbias is not None:
            dbias = dbias[:ctx.weight.shape[0]]
        return dx, dw, dbias
    dw = conv_wgrad(dz, ctx.x, ctx.weight, ctx.stride, ctx.pad) if need_dw else None
    dx = None
    if need_dx and producer is not None and producer.act == K.ACT_LEAKY and producer.a.shape[3] % 16 == 0:
        pb = zeros_f32((2, producer.a.shape[3]), dz.device) if need_dw else None
        pdz = conv_dgrad(dz, ctx.weight, ctx.stride, ctx.pad, ctx.x.shape[1], ctx.x.shape[2], mask=producer.a,
                         mask_slope=producer.slope, dbias=pb)
        dx = (pdz, None if pb is None else pb[0])
    elif need_dx:
        dx = conv_dgrad(dz, ctx.weight, ctx.stride, ctx.pad, ctx.x.shape[1], ctx.x.shape[2])
    if dbias is not None:
        dbias = dbias[:ctx.weight.shape[0]]
    return dx, dw, dbias


# --------------------------------------------------------------------------- global-pool attention
class FcCtx:
    __slots__ = ("inp", "in_scale", "W", "bn", "training", "act", "pre", "out", "mean", "rstd")


def fc_fwd(inp, in_scale, weight, bn, training, act):
    """1x1 conv on an [N, C] vector (+BatchNorm over the batch) + activation."""
    n = inp.shape[0]
    co = weight.shape[0]
    if bn is not None and training and n < 2:
        raise ValueError("Expected more than 1 value per channel when training, got input size [%d, %d, 1, 1]" % (n, co))
    buf = torch.empty((2, n, co), dtype=F32, device=inp.device)
    ms = torch.empty((2, co), dtype=F32, device=inp.device)
    W = weight.detach().view(co, -1)
    K.fc_small_fwd(inp, in_scale, W, bn, training, act, buf[0], buf[1], ms[0], ms[1])
    ctx = FcCtx()
    ctx.inp, ctx.in_scale, ctx.W, ctx.bn, ctx.training, ctx.act = inp, in_scale, W, bn, training, act
    ctx.pre, ctx.out, ctx.mean, ctx.rstd = buf[0], buf[1], ms[0], ms[1]
    return buf[1], ctx


def fc_bwd(ctx, dout, need_din=True):
    """-> (din [N, Cin] (already multiplied by in_scale), dW (conv-shaped), dgamma, dbeta)"""
    n, cin = ctx.inp.shape
    co = ctx.W.shape[0]
    dev = dout.device
    scratch = torch.empty((n, co), dtype=F32, device=dev)
    dW = zeros_f32((co, cin), dev)
    has_bn = ctx.bn is not None
    dgb = zeros_f32((2, co), dev) if has_bn else None
    din = torch.empty((n, cin), dtype=F32, device=dev) if need_din else None
    K.fc_small_bwd(dout, ctx.out, ctx.pre, ctx.inp, ctx.in_scale, ctx.W, has_bn, ctx.training,
                   ctx.bn[0] if has_bn else None, ctx.mean, ctx.rstd, ctx.act, scratch, dW,
                   dgb[0] if has_bn else None, dgb[1] if has_bn else None, din)
    return din, dW.view(co, cin, 1, 1), (dgb[0] if has_bn else None), (dgb[1] if has_bn else None)


def pool_sum(x):
    out = zeros_f32((x.shape[0], x.shape[3]), x.device)
    K.pool_sum(x, out)
    return out


# --------------------------------------------------------------------------- depthwise + BN (+pool)
class DwCtx:
    __slots__ = ("x", "weight", "k", "bn", "z", "a", "act", "slope", "has_pool", "bias")


def dw_bn_fwd(x, weight, bn, training, pool_out=None, act=K.ACT_NONE, slope=0.0, bias=None, out=None):
    """Depthwise k x k stride-2 conv (+ fused 3x3/s2 average pool of the same input) followed by
    BatchNorm (+act).  With bn=None: conv + bias + act only."""
    n, h, w, c = x.shape
    k = weight.shape[2]
    ho, wo = (h + 2 - k) // 2 + 1, (w + 2 - k) // 2 + 1
    wflat = weight.detach().view(-1)
    ctx = DwCtx()
    ctx.x, ctx.weight, ctx.k, ctx.act, ctx.slope, ctx.has_pool, ctx.bias = x, weight, k, act, slope, pool_out is not None, bias
    if bn is not None:
        z = empty_act(n, ho, wo, c, x.device)
        stats = zeros_f32((2, c), x.device) if training else None
        K.dwconv_s2_fwd(x, k, wflat, bias, z, pool_out, K.ACT_NONE, 0.0, stats)
        a, ctx.bn = bn_act_fwd(z, stats, bn, training, act, slope, out)
        ctx.z, ctx.a = z, a
        return a, ctx
    a = empty_act(n, ho, wo, c, x.device)
    K.dwconv_s2_fwd(x, k, wflat, bias, a, pool_out, act, slope, None)
    ctx.bn, ctx.z, ctx.a = None, None, a
    return a, ctx


def dw_bn_bwd(ctx, dy, dpool=None, need_dx=True, dy2=None):
    """-> (dx, dW, dbias, dgamma, dbeta); dy2: a second gradient of the same output, summed in the
    BatchNorm backward pass (BatchNorm'd layers only)."""
    dev = dy.device
    c = ctx.x.shape[3]
    dgamma = dbeta = dbias = None
    if ctx.bn is not None:
        dz, dgamma, dbeta = bn_act_bwd(ctx.bn, dy, dy2)
        if ctx.bias is not None:
            dbias = zeros_f32((c,), dev)
    else:
        dz = torch.empty(ctx.a.shape, dtype=BF16, device=dev)
        dbias = zeros_f32((c,), dev) if ctx.bias is not None else None
        K.act_bwd_bias(dy, dy2, ctx.a, dz, ctx.act, ctx.slope, None)
    dw = zeros_f32((c * ctx.k * ctx.k,), dev)
    K.dwconv_s2_wgrad(dz, ctx.x, ctx.k, dw, dbias)
    dx = None
    if need_dx:
        dx = torch.empty(ctx.x.shape, dtype=BF16, device=dev)
        K.dwconv_s2_dgrad(dz, dpool, ctx.k, ctx.weight.detach().view(-1), dx)
    return dx, dw.view(ctx.weight.shape[0], 1, ctx.k, ctx.k)[: ctx.weight.shape[0]], dbias, dgamma, dbeta


# --------------------------------------------------------------------------- small helpers
def add_acts(a, b, out=None):
    """a + b for two NHWC bf16 views of the same shape (gradient joins of branching features)."""
    if out is None:
        out = torch.empty(a.shape, dtype=BF16, device=a.device)
    K.scale_add_bcast(a, None, 1.0, None, 0.0, b, out)
    return out


def add_bcast_vec(a, v):
    """a[n,h,w,c] + v[n,c]"""
    out = torch.empty(a.shape, dtype=BF16, device=a.device)
    K.scale_add_bcast(a, None, 1.0, v, 1.0, None, out)
    return out


def zeros_act(shape, device):
    return torch.zeros(shape, dtype=BF16, device=device)
