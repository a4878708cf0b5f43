"""Torch-facing wrappers of the C-ABI kernels: torch only provides device memory, the current
stream and autograd bookkeeping; every FLOP and byte below runs in libpixelssl_b200.so.

Conventions
  * backbone activations: logical [N,C,H,W] tensors in ``torch.channels_last`` (physical NHWC);
  * conv weights: logical [Cout,Cin,kh,kw] in channels_last (physical [Cout][kh*kw][Cin]);
  * logit / probability maps (C = num_classes): plain contiguous NCHW ("planar"), as in the
    reference; labels: float [n,1,H,W] holding integers (task/sseg/data.py:179-182).
All tensors must be fp32 CUDA tensors; anything else raises (no silent fallback)."""
import ctypes
import os as _os

import torch

from . import _lib
from ._lib import ConvGeom, ConvTcExt, call

CL = torch.channels_last
# conv precision policy (pxl_conv_geom.precision): 0 fp32 FFMA, 1 TF32 tcgen05, 2 3xTF32 tcgen05,
# 3 fp16-pair x3 tcgen05 (fp32-grade), 4 single fp16 tcgen05 (TF32-grade)
PRECISION = {'fp32': 0, 'tf32': 1, 'tf32x3': 2, 'f16x3': 3, 'f16': 4}
H16_FALLBACK = {3: 2, 4: 1}     # shapes the kind::f16 kernels do not cover run on the tf32 kernels of the same grade
H16_ACT_SCALE = 16.0            # fixed power-of-two scales of fp16 pairs (csrc/h16_prep.cu): activations saturate
H16_W_SCALE = 256.0             # beyond +-4094, weights beyond +-255 (counted: h16_status())
H16_GRAD_TARGET_LOG2 = 14       # gradients: per-tensor scale putting the absmax in (2^13, 2^14]
_conv_precision = 0
_WGRAD_TC_STRIDES = (1, 2)      # convolution strides the tcgen05 wgrad kernel handles


def set_conv_precision(name):
    global _conv_precision
    _conv_precision = PRECISION[name]


def get_conv_precision():
    return _conv_precision


def _p(t):
    """Device address for a C-ABI pointer argument (every entry point declares argtypes, so ctypes converts the
    plain int / None itself: no c_void_p object per argument, ~9000 of them per step)."""
    return t.data_ptr() if t is not None else None


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None)
_cur_device = getattr(torch._C, '_cuda_getDevice', None)


def _stream():
    """Raw handle of torch's current stream.  torch.cuda.current_stream() builds a Stream object through three layers
    of Python (~15 us; ~900 launches per step made that a fifth of the step's host time) - the C accessor is ~0.3 us."""
    if _raw_stream is not None:
        return _raw_stream(_cur_device())
    return torch.cuda.current_stream().cuda_stream


def _chk(t, name, cl=False):
    if getattr(t, '_pxl_carrier', False):
        raise TypeError('%s is an fp16-pair carrier (its storage holds no fp32 values); only conv_bn_act may consume it' % name)
    if not (t.is_cuda and t.dtype == torch.float32):
        raise TypeError('%s must be a CUDA float32 tensor (got %s on %s)' % (name, t.dtype, t.device))
    if cl:
        if t.dim() != 4 or not t.is_contiguous(memory_format=CL):
            raise ValueError('%s must be a 4-D channels_last tensor' % name)
    elif not t.is_contiguous():
        raise ValueError('%s must be contiguous' % name)


def as_cl(t):
    """Return t in channels_last physical layout (no copy if it already is)."""
    return t.contiguous(memory_format=CL)


_workspaces = {}
_ktimers = {}


def kernel_timer_start(name):
    """Record CUDA events (on the launching stream) around every subsequent launch of the named
    entry point; bench.py uses it to time the metric kernel inside the timed steps."""
    _ktimers[name] = []


def kernel_timer_stop(name, with_meta=False):
    """-> per-launch milliseconds; with_meta: [(ms, meta)] where meta is what the call site attached (the
    algorithmic FLOPs of a convolution launch)."""
    pairs = _ktimers.pop(name, [])
    torch.cuda.synchronize()
    if with_meta:
        return [(a.elapsed_time(b), m) for a, b, m in pairs]
    return [a.elapsed_time(b) for a, b, _ in pairs]


def _timed_call(name, *args, meta=None):
    rec = _ktimers.get(name)
    if rec is None:
        return call(name, *args)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    rc = call(name, *args)
    b.record()
    rec.append((a, b, meta))
    return rc


def _mse_ws(device):
    ws = _workspaces.get(device)
    if ws is None:
        n = _lib.load().pxl_mse_workspace_bytes()
        ws = torch.zeros((n + 7) // 8, dtype=torch.float64, device=device)
        _workspaces[device] = ws
    return ws


# ------------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------------

def mse_consistency_raw(s, t, loss_scale=1.0, want_grad=True):
    """Fused forward(+backward) of loss_scale * mean((s-t)^2).  Returns (loss[1], grad or None)."""
    _chk(s, 's'); _chk(t, 't')
    if s.shape != t.shape:
        raise ValueError('shape mismatch')
    loss = torch.empty(1, dtype=torch.float32, device=s.device)
    grad = torch.empty_like(s) if want_grad else None
    _timed_call('pxl_mse_consistency', _p(s), _p(t), s.numel(), float(loss_scale), _p(loss), _p(grad),
                _p(_mse_ws(s.device)), _stream())
    return loss, grad


class _MseConsistency(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, t, loss_scale, unit_upstream):
        need = ctx.needs_input_grad[0]
        loss, grad = mse_consistency_raw(s, t, loss_scale, want_grad=need and unit_upstream)
        ctx.unit, ctx.scale = unit_upstream, loss_scale
        if need:
            if unit_upstream:
                ctx.save_for_backward(grad)
            else:
                ctx.save_for_backward(s, t)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        if ctx.unit:
            (grad,) = ctx.saved_tensors
            return grad, None, None, None
        s, t = ctx.saved_tensors
        grad = torch.empty_like(s)
        g = g.reshape(1).contiguous().float()
        call('pxl_mse_consistency_bwd', _p(s), _p(t), s.numel(), float(ctx.scale), _p(g), _p(grad), _stream())
        return grad, None, None, None


def mse_consistency(s, t, loss_scale=1.0, unit_upstream=False):
    """nn.MSELoss()(s, t.detach()) * loss_scale (ssl_mt.py:115,179-187).

    unit_upstream=True: the caller guarantees the returned scalar is added, un-scaled, into the
    loss on which ``backward()`` is called (d total / d this = 1), so the gradient is produced by
    the same kernel launch as the loss (12 B/element instead of 8 + 12)."""
    return _MseConsistency.apply(s.contiguous(), t.detach().contiguous(), float(loss_scale), bool(unit_upstream))


def _labels_flat(gt, n, hw):
    if gt.numel() != n * hw:
        raise ValueError('label tensor has %d elements, expected %d' % (gt.numel(), n * hw))
    _chk(gt, 'gt')
    return gt


class _CrossEntropy2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, gt, ignore_index, upstream_const):
        _chk(logits, 'logits')
        n, c, h, w = logits.shape
        gt = _labels_flat(gt, n, h * w)
        per = torch.empty(n, dtype=torch.float32, device=logits.device)
        need = ctx.needs_input_grad[0]
        fused = need and upstream_const is not None
        grad = torch.empty_like(logits) if fused else None
        call('pxl_ce2d', _p(logits), _p(gt), n, c, h * w, int(ignore_index), _p(per), _p(grad),
             _p(None), float(upstream_const or 0.0), _stream())
        ctx.fused, ctx.ignore = fused, int(ignore_index)
        if need:
            if fused:
                ctx.save_for_backward(grad)
            else:
                ctx.save_for_backward(logits, gt)
        return per

    @staticmethod
    def backward(ctx, g):
        if ctx.fused:
            (grad,) = ctx.saved_tensors
            return grad, None, None, None
        logits, gt = ctx.saved_tensors
        n, c, h, w = logits.shape
        per = torch.empty(n, dtype=torch.float32, device=logits.device)
        grad = torch.empty_like(logits)
        g = g.contiguous().float()
        call('pxl_ce2d', _p(logits), _p(gt), n, c, h * w, ctx.ignore, _p(per), _p(grad), _p(g), 0.0, _stream())
        return grad, None, None, None


def cross_entropy2d(logits, gt, ignore_index=255, upstream_const=None):
    """CommonSSEGCriterion.forward (task/sseg/criterion.py:24-38) -> per-sample loss [n].

    upstream_const: if given, the caller guarantees d total / d per_sample[i] == upstream_const
    (e.g. 1/n when ``torch.mean`` of the result goes straight into the loss) and the gradient is
    written by the forward launch."""
    return _CrossEntropy2d.apply(logits.contiguous(), gt.contiguous(), ignore_index, upstream_const)


class _Softmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits):
        _chk(logits, 'logits')
        n, c, h, w = logits.shape
        prob = torch.empty_like(logits)
        call('pxl_softmax_planar', _p(logits), _p(prob), n, c, h * w, _stream())
        ctx.save_for_backward(prob)
        return prob

    @staticmethod
    def backward(ctx, g):
        (prob,) = ctx.saved_tensors
        n, c, h, w = prob.shape
        g = g.contiguous()
        out = torch.empty_like(prob)
        call('pxl_softmax_planar_bwd', _p(prob), _p(g), _p(out), n, c, h * w, _stream())
        return out


def softmax_planar(logits):
    """F.softmax(pred, dim=1) on a planar map (task/sseg/model.py:62)."""
    return _Softmax.apply(logits.contiguous())


class _SoftmaxMse(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, tprob, loss_scale):
        _chk(logits, 'logits'); _chk(tprob, 'tprob')
        n, c, h, w = logits.shape
        loss = torch.empty(1, dtype=torch.float32, device=logits.device)
        need = ctx.needs_input_grad[0]
        grad = torch.empty_like(logits) if need else None
        call('pxl_softmax_mse', _p(logits), _p(tprob), n, c, h * w, float(loss_scale), _p(loss), _p(None),
             _p(grad), _p(_mse_ws(logits.device)), _stream())
        if need:
            ctx.save_for_backward(grad)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None, None


def softmax_mse(logits, tprob, loss_scale=1.0):
    """loss_scale * MSE(softmax(logits), tprob) with the gradient through the softmax produced in
    the same pass (ssl_cutmix.py:206-215).  Backward multiplies by the upstream scalar."""
    return _SoftmaxMse.apply(logits.contiguous(), tprob.detach().contiguous(), float(loss_scale))


def cutmix_mix(mask, a, b):
    """mask*a + (1-mask)*b, bit-exact with the reference's fp32 op order (ssl_cutmix.py:195,428).
    mask: [n,1,H,W]; a, b: [n,C,H,W] planar."""
    _chk(mask, 'mask'); _chk(a, 'a'); _chk(b, 'b')
    n, c, h, w = a.shape
    out = torch.empty_like(a)
    call('pxl_cutmix_mix', _p(mask), _p(a), _p(b), _p(out), n, c, h * w, _stream())
    return out


def cutmix_confidence(prob, thr):
    """mean(max_c p > thr) over the batch as a device scalar (ssl_cutmix.py:200)."""
    _chk(prob, 'prob')
    n, c, h, w = prob.shape
    cnt = torch.empty(1, dtype=torch.int64, device=prob.device)
    call('pxl_cutmix_confidence', _p(prob), n, c, h * w, float(thr), _p(cnt), _stream())
    return (cnt.to(torch.float64).reshape(()) / float(n * h * w)).to(torch.float32)   # correctly rounded count/N


# ------------------------------------------------------------------------------------------------
# bilinear resize
# ------------------------------------------------------------------------------------------------

class _Bilinear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, C, size, align_corners, in_nhwc):
        H, W = size
        if in_nhwc:
            _chk(x, 'x', cl=True)
            n, ldc, h, w = x.shape
        else:
            _chk(x, 'x')
            n, ldc, h, w = x.shape
            if ldc != C:
                raise ValueError('planar input must have exactly C channels')
        out = torch.empty((n, C, H, W), dtype=torch.float32, device=x.device)
        call('pxl_bilinear_fwd', _p(x), _p(out), n, C, h, w, H, W, int(align_corners), int(in_nhwc), ldc, _stream())
        ctx.meta = (n, C, h, w, H, W, int(align_corners), int(in_nhwc), ldc)
        return out

    @staticmethod
    def backward(ctx, g):
        n, C, h, w, H, W, ac, nhwc, ldc = ctx.meta
        g = g.contiguous()
        if nhwc:
            gin = torch.empty((n, ldc, h, w), dtype=torch.float32, device=g.device, memory_format=CL).zero_()
        else:
            gin = torch.empty((n, C, h, w), dtype=torch.float32, device=g.device)
        call('pxl_bilinear_bwd', _p(g), _p(gin), n, C, h, w, H, W, ac, nhwc, ldc, _stream())
        return gin, None, None, None, None


def bilinear(x, size, align_corners=True, channels=None, nhwc=False):
    """F.interpolate(x, size, mode='bilinear', align_corners) -> planar [n,C,H,W].
    nhwc=False: x planar [n,C,h,w].  nhwc=True: x channels_last [n,ldc,h,w] of which the first
    ``channels`` (<= ldc) channels are real (e.g. the 32-lane padded ASPP output)."""
    if channels is None:
        channels = x.shape[1]
    x = as_cl(x) if nhwc else x.contiguous()
    return _Bilinear.apply(x, int(channels), (int(size[0]), int(size[1])), bool(align_corners), bool(nhwc))


# ------------------------------------------------------------------------------------------------
# convolution
# ------------------------------------------------------------------------------------------------

def _taps(kh, kw, dil, pad):
    t = []
    for r in range(kh):
        for s in range(kw):
            t += [r * dil - pad, s * dil - pad]
    return t


def _ctaps(t):
    return (ctypes.c_int * len(t))(*t)


_epoch = 0
ACCUM_WGRAD_INPLACE = True      # wgrad kernels add straight into weight.grad (the flat gradient arena)
FUSE_BN_FINALIZE = _os.environ.get('PXL_BN_FUSED_FINALIZE', '1') != '0'     # finalize inside the apply launch
BATCH_WEIGHT_PREP = _os.environ.get('PXL_BATCH_WEIGHT_PREP', '1') != '0'    # arena-wide weight transposes / tf32 splits


def new_step():
    """Called once per training step: invalidates the cached tf32 splits of the weights (the fused
    SGD kernel updates parameters through raw pointers, invisible to torch's version counters) and
    recycles the statistics pool."""
    global _epoch
    _epoch += 1
    _stat_pool_reset()
    _residual_stash.clear()


# Per-channel fp64 accumulators (BN sums, their gradients) are tiny and short-lived (consumed by the next
# launch on the same stream); carving them out of one pool that is cleared with ONE memset per step
# replaces ~300 two-kilobyte memsets per MT step.
_STAT_POOL_DOUBLES = 1 << 20
_stat_pool = {}


def _stat_zeros(n, device):
    ent = _stat_pool.get(device)
    if ent is None:
        ent = _stat_pool[device] = [torch.zeros(_STAT_POOL_DOUBLES, dtype=torch.float64, device=device), 0]
    buf, cur = ent
    n_al = (n + 1) & ~1                              # keep 16-byte alignment
    if cur + n_al > buf.numel():
        return torch.zeros(n, dtype=torch.float64, device=device)
    ent[1] = cur + n_al
    return buf[cur:cur + n]


def _stat_pool_reset():
    for ent in _stat_pool.values():
        if ent[1]:
            ent[0][:ent[1]].zero_()
            ent[1] = 0


def step_epoch():
    return _epoch


# parameter arenas (nn/arena.py) register here so that per-layer requests for a split / transposed weight can be
# served from the arena-wide copies made with one launch per step
_param_arenas = []


def register_param_arena(arena):
    import weakref
    _param_arenas.append(weakref.ref(arena))


def _arena_of(t):
    for ref in list(_param_arenas):
        a = ref()
        if a is None:
            _param_arenas.remove(ref)
            continue
        off = a.locate(t)
        if off is not None:
            return a, off
    return None, None


def transpose_weights_batched(src, dst, table, total_tiles):
    call('pxl_conv_transpose_weights_batched', _p(src), _p(dst), ctypes.c_void_p(table.data_ptr()), int(table.shape[0]),
         int(total_tiles), _stream())


def split_tf32_into(x, hi, lo):
    call('pxl_split_tf32', _p(x), _p(hi), _p(lo), x.numel(), _stream())


def split_tf32(x):
    """x (any shape, numel % 4 == 0) -> (hi, lo): hi = tf32(x) with a zero low mantissa, lo = x - hi."""
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    call('pxl_split_tf32', _p(x), _p(hi), _p(lo), x.numel(), _stream())
    return hi, lo


def split_cached(x):
    """split_tf32 memoised on the tensor object (an activation feeding two convolutions, a weight
    used by several launches of one step).  Invalidated by in-place edits and by new_step()."""
    arena, off = _arena_of(x) if (x.dim() == 4 and BATCH_WEIGHT_PREP) else (None, None)
    if arena is not None and off in arena._conv_at:
        n = x.numel()
        return arena.derived('hi')[off:off + n], arena.derived('lo')[off:off + n]
    ent = getattr(x, '_pxl_parts', None)
    if ent is not None and ent[0] == _epoch and ent[1] == x._version and ent[2] == x.data_ptr():
        return ent[3]
    parts = split_tf32(x)
    try:
        x._pxl_parts = (_epoch, x._version, x.data_ptr(), parts)
    except Exception:
        pass
    return parts


class H16:
    """fp16 pair of a tensor (csrc/h16_prep.cu): ``buf`` = [2, numel] half (hi plane, lo plane; ``lo`` is None in
    single-fp16 mode), value * scale = hi + lo.  ``scale`` is the fixed power of two, or None when the scale is
    dynamic and lives on the device in ``slot`` ([s, 1/s, absmax bits, -])."""
    __slots__ = ('buf', 'numel', 'scale', 'slot', 'has_lo')

    def __init__(self, buf, numel, scale, slot, has_lo):
        self.buf, self.numel, self.scale, self.slot, self.has_lo = buf, numel, scale, slot, has_lo

    @property
    def hi(self):
        return self.buf[0]

    @property
    def lo(self):
        return self.buf[1] if self.has_lo else None

    @property
    def device(self):
        return self.buf.device

    def inv_scale(self):
        """(host factor, device pointer or None) undoing this operand's scale in a consumer's epilogue."""
        if self.slot is None:
            return 1.0 / self.scale, None
        return 1.0, self.slot[1:]


def _scale_slot(device):
    """A zeroed device float[4] carved out of the per-step statistics pool."""
    return _stat_zeros(2, device).view(torch.float32)


def h16_split(x, scale=None, want_lo=True):
    """fp32 tensor (any layout, numel % 4 == 0) -> H16.  scale None: dynamic (absmax pass + split)."""
    n = x.numel()
    buf = torch.empty((2 if want_lo else 1, n), dtype=torch.float16, device=x.device)
    slot = None
    if scale is None:
        slot = _scale_slot(x.device)
        call('pxl_h16_absmax', _p(x), n, _p(slot), _stream())
    call('pxl_h16_split', _p(x), _p(buf[0]), _p(buf[1] if want_lo else None), n, float(scale or 1.0), _p(slot),
         H16_GRAD_TARGET_LOG2, _stream())
    return H16(buf, n, scale, slot, want_lo)


def h16_status():
    """Number of fp16-pair producers that saturated since the last reset (0 = every operand was in range)."""
    return int(_lib.load().pxl_h16_status())


def h16_status_sites():
    """Saturation events per producer: (split fixed, split dynamic, BN apply, BN backward dx)."""
    out = (ctypes.c_int * 4)()
    _lib.load().pxl_h16_status_sites(out)
    return tuple(int(v) for v in out)


def h16_cached(x, scale, want_lo=True):
    """h16_split memoised on the tensor object for one step (a weight used by several launches)."""
    ent = getattr(x, '_pxl_h16', None)
    if ent is not None and ent[0] == _epoch and ent[1] == x._version and ent[2] == x.data_ptr() and ent[3].has_lo >= want_lo:
        return ent[3]
    h = h16_split(x, scale, want_lo)
    try:
        x._pxl_h16 = (_epoch, x._version, x.data_ptr(), h)
    except Exception:
        pass
    return h


def h16_weight(w, transposed_of=None):
    """fp16 pair of a packed conv weight; arena weights are served from the arena-wide pair made once per step."""
    want_lo = _conv_precision == 3
    arena, off = _arena_of(w) if (w.dim() == 4 and BATCH_WEIGHT_PREP) else (None, None)
    if arena is not None and off in arena._conv_at:
        n = w.numel()
        return H16(arena.derived('h16')[:, off:off + n], n, H16_W_SCALE, None, True)
    return h16_cached(w, H16_W_SCALE, want_lo)


def h16_supported(Cin, mul, div):
    return Cin % 64 == 0 and ((div == 1 and mul in (1, 2)) or (div == 2 and mul == 1))


def tc_supported(Cin, mul, div):
    """Shapes covered by the tcgen05 forward/dgrad kernel (csrc/conv_tc.cu): stride 1 and 2 forward
    (mul), and the dgrad of a stride-2 convolution (div == 2, decomposed by output parity)."""
    return Cin % 32 == 0 and ((div == 1 and mul in (1, 2)) or (div == 2 and mul == 1))


def _stride2_dgrad_classes(taps, ntaps):
    """dgrad of a stride-2 convolution: output pixel (iy, ix) only receives the taps with (iy + dy) and (ix + dx)
    even; per output parity class that is a stride-1 problem over dY.  -> [(py, px, halved taps, tap indices)]"""
    classes = []
    for py in (0, 1):
        for px in (0, 1):
            sub, widx = [], []
            for t in range(ntaps):
                dy, dx = taps[2 * t], taps[2 * t + 1]
                if (py + dy) % 2 == 0 and (px + dx) % 2 == 0:
                    sub += [(py + dy) // 2, (px + dx) // 2]
                    widx.append(t)
            classes.append((py, px, sub, widx))
    return classes


def _tc_launch(geom, taps, ext, x_parts, w_parts, bias, out):
    _timed_call('pxl_conv_tc_launch_ex', ctypes.byref(geom), _ctaps(taps), ctypes.byref(ext) if ext is not None else None,
                _p(x_parts[0]), _p(x_parts[1]), _p(w_parts[0]), _p(w_parts[1]), _p(bias), _p(out), _stream(),
                meta=(2.0 * geom.N * geom.OH * geom.OW * geom.Cin * geom.Cout * geom.ntaps,
                      'fwd/dgrad(tf32) N%d %dx%d Cin%d Cout%d taps%d' % (geom.N, geom.OH, geom.OW, geom.Cin, geom.Cout, geom.ntaps)))


def conv_raw(x, w_packed, bias, taps, N, H, W, Cin, OH, OW, Cout, ldo, mul, div, out=None, precision=None, bn_stats=None,
             accumulate=False):
    """Launch the NHWC tap-table convolution on raw buffers.  w_packed: [Cout][ntaps][Cin] contiguous.
    precision 0: FFMA kernel; 1: tcgen05 single-pass TF32; 2: tcgen05 3xTF32 (operands split on the
    fly).  Shapes the tensor-core kernel does not cover (Cin % 32 != 0, other strides) use the FFMA kernel."""
    ntaps = len(taps) // 2
    prec = _conv_precision if precision is None else precision
    if out is None and not isinstance(x, H16):
        dev = x[0].device if isinstance(x, tuple) else x.device
        out = torch.empty((N, ldo, OH, OW), dtype=torch.float32, device=dev, memory_format=CL)
        if ldo != Cout:
            out.zero_()
    if prec >= 3 and not h16_supported(Cin, mul, div):
        if isinstance(x, H16) or isinstance(w_packed, H16):
            raise ValueError('fp16-pair operands given for a shape the kind::f16 kernel does not cover')
        prec = H16_FALLBACK[prec]
    if prec >= 3:
        want_lo = prec == 3
        xh = x if isinstance(x, H16) else h16_cached(x, H16_ACT_SCALE, want_lo)
        wh = w_packed if isinstance(w_packed, H16) else h16_weight(w_packed)
        fx, px = xh.inv_scale()
        fw, pw = wh.inv_scale()
        if px is not None and pw is not None:
            raise ValueError('at most one operand may carry a device-side scale')
        oscale, odev = fx * fw, (px if px is not None else pw)
        if out is None:
            out = torch.empty((N, ldo, OH, OW), dtype=torch.float32, device=xh.device, memory_format=CL)
            if ldo != Cout:
                out.zero_()

        def launch(geom, tp, ext):
            ext.out_scale, ext.out_scale_dev = oscale, (odev.data_ptr() if odev is not None else None)
            ext.out_accumulate = 1 if accumulate else 0
            _timed_call('pxl_conv_h16_launch', ctypes.byref(geom), _ctaps(tp), ctypes.byref(ext), _p(xh.hi), _p(xh.lo),
                        _p(wh.hi), _p(wh.lo if want_lo else None), _p(bias), _p(out), _stream(),
                        meta=(2.0 * geom.N * geom.OH * geom.OW * geom.Cin * min(geom.Cout, Cout) * geom.ntaps,
                              'fwd/dgrad N%d %dx%d Cin%d Cout%d taps%d mul%d' % (geom.N, geom.OH, geom.OW, geom.Cin, geom.Cout, geom.ntaps, geom.mul)))
        if div == 1:
            ext = ConvTcExt(0, None, 0, 0, 0, 0, 0, None)
            if bn_stats is not None:
                ext.bn_stats = bn_stats.data_ptr()
                bn_stats._pxl_filled = True
            launch(ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, 1, ntaps, prec), taps, ext)
            return out
        classes = _stride2_dgrad_classes(taps, ntaps)
        if any(len(c[3]) == 0 for c in classes):
            out.zero_()
        for py, px_, sub, widx in classes:
            ohs, ows = (OH - py + 1) // 2, (OW - px_ + 1) // 2
            if not widx or ohs <= 0 or ows <= 0:
                continue
            ext = ConvTcExt(ntaps, (ctypes.c_int * len(widx))(*widx), 2, py, px_, OH, OW, None)
            launch(ConvGeom(N, H, W, Cin, ohs, ows, Cout, ldo, 1, 1, len(widx), prec), sub, ext)
        return out
    if prec != 0 and tc_supported(Cin, mul, div):
        if prec == 2:
            # activations go in raw: the kernel splits them hi/lo in shared memory; the (small, per-step
            # cached) weights are split here
            x_parts = x if isinstance(x, tuple) else (x, None)
            w_parts = w_packed if isinstance(w_packed, tuple) else split_cached(w_packed)
        else:
            x_parts, w_parts = (x, None), (w_packed, None)
        if div == 1:
            geom = ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, 1, ntaps, prec)
            ext = None
            if bn_stats is not None:      # the epilogue also accumulates sum(y), sum(y^2) per channel
                ext = ConvTcExt(0, None, 0, 0, 0, 0, 0, ctypes.c_void_p(bn_stats.data_ptr()))
                bn_stats._pxl_filled = True
            _tc_launch(geom, taps, ext, x_parts, w_parts, bias, out)
            return out
        classes = _stride2_dgrad_classes(taps, ntaps)
        if any(len(c[3]) == 0 for c in classes):
            out.zero_()
        for py, px, sub, widx in classes:
            ohs, ows = (OH - py + 1) // 2, (OW - px + 1) // 2
            if not widx or ohs <= 0 or ows <= 0:
                continue
            geom = ConvGeom(N, H, W, Cin, ohs, ows, Cout, ldo, 1, 1, len(widx), prec)
            ext = ConvTcExt(ntaps, (ctypes.c_int * len(widx))(*widx), 2, py, px, OH, OW, None)
            _tc_launch(geom, sub, ext, x_parts, w_parts, bias, out)
        return out
    if isinstance(x, tuple):
        x = x[0] + x[1]
    if isinstance(w_packed, tuple):
        w_packed = w_packed[0] + w_packed[1]
    geom = ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, div, ntaps, 0)
    call('pxl_conv_nhwc', ctypes.byref(geom), _ctaps(taps), _p(x), _p(w_packed), _p(bias), _p(out), _stream())
    return out


def conv_tc_status():
    """0 when every tcgen05 pipeline so far completed; otherwise the role whose mbarrier wait timed out."""
    return int(_lib.load().pxl_conv_tc_status())


_wgrad_ws = {}          # (device, stream) -> workspace of the tcgen05 wgrad launches enqueued on that stream
_wgrad_ws_need = {}     # geometry -> floats it needs


def _wgrad_workspace(geom, taps, device, key):
    """Workspace of one tcgen05 wgrad launch (its per-split dW slots).  One per stream, so that launches on different
    streams never share slots; a larger request replaces it through torch's caching allocator, which hands the old
    block out again only after the work already queued on that stream."""
    need = _wgrad_ws_need.get(key)
    if need is None:
        need = int(_lib.load().pxl_conv_wgrad_workspace_floats(ctypes.byref(geom), _ctaps(taps)))
        if need < 0:
            raise _lib.PxlError('pxl_conv_wgrad_workspace_floats', need)
        _wgrad_ws_need[key] = need
    skey = (device, _stream())
    ws = _wgrad_ws.get(skey)
    if ws is None or ws.numel() < need:
        ws = _wgrad_ws[skey] = torch.empty(need, dtype=torch.float32, device=device)
    return ws


def conv_wgrad_raw(x, dy, dw, taps, N, H, W, Cin, OH, OW, Cout, ldo, mul, div, precision=None):
    """dw[Cout][ntaps][Cin] += ...  (dw must be initialised by the caller)."""
    ntaps = len(taps) // 2
    prec = _conv_precision if precision is None else precision
    if prec >= 3 and not (div == 1 and mul in _WGRAD_TC_STRIDES and Cin % 64 == 0 and ldo % 64 == 0):
        if isinstance(x, H16) or isinstance(dy, H16):
            raise ValueError('fp16-pair operands given for a shape the kind::f16 wgrad kernel does not cover')
        prec = H16_FALLBACK[prec]
    if prec >= 3:
        want_lo = prec == 3
        xh = x if isinstance(x, H16) else h16_split(x, H16_ACT_SCALE, want_lo)
        dh = dy if isinstance(dy, H16) else h16_split(dy, None, want_lo)
        fx, px = xh.inv_scale()
        fd, pd = dh.inv_scale()
        if px is not None and pd is not None:
            raise ValueError('at most one operand may carry a device-side scale')
        geom = ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, div, ntaps, prec)
        ws = _wgrad_workspace(geom, taps, dw.device, (N, H, W, Cin, OH, OW, Cout, ldo, mul, div, prec, tuple(taps)))
        _timed_call('pxl_conv_wgrad_h16_launch', ctypes.byref(geom), _ctaps(taps), _p(xh.hi), _p(xh.lo), _p(dh.hi), _p(dh.lo),
                    _p(dw), float(fx * fd), _p(pd if pd is not None else px), _p(ws), ws.numel(), _stream(),
                    meta=(2.0 * N * OH * OW * Cin * Cout * ntaps, 'wgrad N%d %dx%d Cin%d Cout%d taps%d mul%d' % (N, OH, OW, Cin, Cout, ntaps, mul)))
        return dw
    if prec != 0 and div == 1 and mul in _WGRAD_TC_STRIDES and Cin % 32 == 0 and ldo % 32 == 0:
        geom = ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, div, ntaps, prec)
        ws = _wgrad_workspace(geom, taps, dw.device, (N, H, W, Cin, OH, OW, Cout, ldo, mul, div, prec, tuple(taps)))
        if prec == 2:
            if isinstance(x, tuple) != isinstance(dy, tuple):        # mixed: split the raw one too
                x = x if isinstance(x, tuple) else split_tf32(x)
                dy = dy if isinstance(dy, tuple) else split_tf32(dy)
            x_hi, x_lo = x if isinstance(x, tuple) else (x, None)     # raw operands: split inside the kernel
            d_hi, d_lo = dy if isinstance(dy, tuple) else (dy, None)
            _timed_call('pxl_conv_wgrad_tc_launch', ctypes.byref(geom), _ctaps(taps), _p(x_hi), _p(x_lo), _p(d_hi), _p(d_lo),
                        _p(dw), _p(ws), ws.numel(), _stream(), meta=(2.0 * N * OH * OW * Cin * Cout * ntaps, 'wgrad(tf32) N%d %dx%d Cin%d Cout%d taps%d' % (N, OH, OW, Cin, Cout, ntaps)))
        else:
            _timed_call('pxl_conv_wgrad_tc_launch', ctypes.byref(geom), _ctaps(taps), _p(x), _p(None), _p(dy), _p(None),
                        _p(dw), _p(ws), ws.numel(), _stream(), meta=(2.0 * N * OH * OW * Cin * Cout * ntaps, 'wgrad(tf32) N%d %dx%d Cin%d Cout%d taps%d' % (N, OH, OW, Cin, Cout, ntaps)))
        return dw
    if isinstance(x, tuple):
        x = x[0] + x[1]
    if isinstance(dy, tuple):
        dy = dy[0] + dy[1]
    geom = ConvGeom(N, H, W, Cin, OH, OW, Cout, ldo, mul, div, ntaps, 0)     # FFMA split-K kernel
    call('pxl_conv_wgrad_nhwc', ctypes.byref(geom), _ctaps(taps), _p(x), _p(dy), _p(dw), _stream())
    return dw


def transpose_weights(w_packed, Cout, T, Cin):
    wt = torch.empty(Cin * T * Cout, dtype=torch.float32, device=w_packed.device)
    call('pxl_conv_transpose_weights', _p(w_packed), _p(wt), Cout, T, Cin, _stream())
    return wt


class _Conv2d(torch.autograd.Function):
    """nn.Conv2d on NHWC (resnet.py:18-25 etc.).  weight logical [Cout,Cin,kh,kw] channels_last."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride, padding, dilation, out_lanes=0, bn_stats=None):
        _chk(x, 'x', cl=True); _chk(weight, 'weight', cl=True)
        N, Cin, H, W = x.shape
        Cout, Cin2, kh, kw = weight.shape
        if out_lanes and out_lanes > Cout:
            return _Conv2d._forward_padded(ctx, x, weight, bias, stride, padding, dilation, out_lanes)
        ctx.padded = False
        if Cin2 != Cin:
            raise ValueError('channel mismatch')
        OH = (H + 2 * padding - dilation * (kh - 1) - 1) // stride + 1
        OW = (W + 2 * padding - dilation * (kw - 1) - 1) // stride + 1
        taps = _taps(kh, kw, dilation, padding)
        ctx.split, ctx.h16 = False, None
        ctx.meta = (taps, N, H, W, Cin, OH, OW, Cout, stride, kh * kw, bias is not None)
        if _conv_precision >= 3 and h16_supported(Cin, stride, 1):
            # fp16-pair path: the pair of x (4 B/element, like x itself) is what the backward keeps
            xh = h16_cached(x, H16_ACT_SCALE, _conv_precision == 3)
            out = conv_raw(xh, weight, bias, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1, bn_stats=bn_stats)
            wg_ok = Cin % 64 == 0 and Cout % 64 == 0 and stride in _WGRAD_TC_STRIDES
            if wg_ok or not ctx.needs_input_grad[1]:
                ctx.save_for_backward(xh.buf, weight)
                ctx.h16 = (xh.scale, xh.has_lo)
            else:
                ctx.save_for_backward(x, weight)
            return out
        out = conv_raw(x, weight, bias, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1, bn_stats=bn_stats)
        ctx.save_for_backward(x, weight)
        return out

    @staticmethod
    def _forward_padded(ctx, x, weight, bias, stride, padding, dilation, ldo):
        """Output written with ``ldo`` > Cout channel lanes (extra lanes zero) so that the consumer can be
        a tensor-core convolution with Cin % 32 == 0.  Used by the 21-channel decoder heads."""
        N, Cin, H, W = x.shape
        Cout, _, kh, kw = weight.shape
        OH = (H + 2 * padding - dilation * (kh - 1) - 1) // stride + 1
        OW = (W + 2 * padding - dilation * (kw - 1) - 1) // stride + 1
        taps = _taps(kh, kw, dilation, padding)
        out = conv_raw(x, weight, bias, taps, N, H, W, Cin, OH, OW, Cout, ldo, stride, 1)
        ctx.save_for_backward(x, weight)
        ctx.padded, ctx.split = True, False
        ctx.meta = (taps, N, H, W, Cin, OH, OW, Cout, stride, kh * kw, bias is not None, ldo)
        return out

    @staticmethod
    def _backward_padded(ctx, dy):
        x, weight = ctx.saved_tensors
        taps, N, H, W, Cin, OH, OW, Cout, stride, T, has_bias, ldo = ctx.meta
        dy = as_cl(dy)                       # [N, ldo, OH, OW]; lanes >= Cout carry zeros
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wp = torch.zeros((ldo, T, Cin), dtype=torch.float32, device=dy.device)
            wp[:Cout] = weight.permute(0, 2, 3, 1).reshape(Cout, T, Cin)
            wt = transpose_weights(wp, ldo, T, Cin)
            dx = conv_raw(dy, wt, None, [-v for v in taps], N, OH, OW, ldo, H, W, Cin, Cin, 1, stride)
        if ctx.needs_input_grad[1]:
            dwp = torch.zeros((Cout, T, Cin), dtype=torch.float32, device=dy.device)
            conv_wgrad_raw(x, dy, dwp, taps, N, H, W, Cin, OH, OW, Cout, ldo, stride, 1)
            kh = int(round(T ** 0.5))
            dw = dwp.reshape(Cout, kh, T // kh, Cin).permute(0, 3, 1, 2)
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(Cout, dtype=torch.float32, device=dy.device)
            call('pxl_bias_grad', _p(dy), N * OH * OW, Cout, ldo, _p(db), 0, _stream())
        return dx, dw, db, None, None, None, None, None

    @staticmethod
    def backward(ctx, dy):
        if ctx.padded:
            return _Conv2d._backward_padded(ctx, dy)
        if ctx.split:
            x_hi, x_lo, weight = ctx.saved_tensors
            x = (x_hi, x_lo)
        else:
            x, weight = ctx.saved_tensors
        taps, N, H, W, Cin, OH, OW, Cout, stride, T, has_bias = ctx.meta
        dy = as_cl(dy)
        dx = dw = db = None
        dyin = dy
        if ctx.h16 is not None:
            x = H16(x, x.shape[1], ctx.h16[0], None, ctx.h16[1])
        prec = _conv_precision
        if prec >= 3:
            dgrad_h16 = ctx.needs_input_grad[0] and h16_supported(Cout, 1, stride)
            wgrad_h16 = ctx.needs_input_grad[1] and isinstance(x, H16)
            if dgrad_h16 or wgrad_h16:
                dyin = h16_split(dy, None, prec == 3)        # one pair of dY serves dgrad and wgrad
        eff = H16_FALLBACK.get(prec, prec)
        if ctx.needs_input_grad[0]:
            want_split = eff == 2 and tc_supported(Cout, 1, stride)
            arena, off = _arena_of(weight) if BATCH_WEIGHT_PREP else (None, None)
            if isinstance(dyin, H16) and h16_supported(Cout, 1, stride):
                if arena is not None and arena._conv_at.get(off) == (Cout, T, Cin):
                    n = weight.numel()
                    wt = H16(arena.derived('h16_t')[:, off:off + n], n, H16_W_SCALE, None, True)
                else:
                    wt = h16_split(transpose_weights(weight, Cout, T, Cin), H16_W_SCALE, prec == 3)
            elif arena is not None and arena._conv_at.get(off) == (Cout, T, Cin):
                n = weight.numel()          # arena-wide transposed (and split) copies: one launch per step each
                if want_split:
                    wt = (arena.derived('t_hi')[off:off + n], arena.derived('t_lo')[off:off + n])
                else:
                    wt = arena.derived('t')[off:off + n]
            elif want_split:
                w_hi, w_lo = split_cached(weight)
                wt = (transpose_weights(w_hi, Cout, T, Cin), transpose_weights(w_lo, Cout, T, Cin))
            else:
                wt = transpose_weights(weight, Cout, T, Cin)
            ntaps = [-v for v in taps]
            dgrad_in = dyin if (isinstance(dyin, H16) and isinstance(wt, H16)) else dy
            dx = conv_raw(dgrad_in, wt, None, ntaps, N, OH, OW, Cout, H, W, Cin, Cin, 1, stride)
        if ctx.needs_input_grad[1]:
            inplace = ACCUM_WGRAD_INPLACE and weight.grad is not None and weight.grad.is_contiguous(memory_format=CL)
            dwbuf = weight.grad if inplace else torch.zeros_like(weight, memory_format=torch.preserve_format)
            conv_wgrad_raw(x, dyin if isinstance(x, H16) else dy, dwbuf, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1)
            dw = None if inplace else dwbuf
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(Cout, dtype=torch.float32, device=dy.device)
            call('pxl_bias_grad', _p(dy), N * OH * OW, Cout, Cout, _p(db), 0, _stream())
        return dx, dw, db, None, None, None, None, None


def conv2d(x, weight, bias=None, stride=1, padding=0, dilation=1, out_lanes=0, want_bn_stats=False):
    """out_lanes > Cout: the output tensor gets that many channel lanes (the extra ones zero).
    want_bn_stats: when the tensor-core kernel runs, its epilogue also accumulates the per-channel
    sum / sum of squares of the output; they are attached to the result as ``._pxl_bn_sums`` (fp64 [2*Cout])
    and picked up by bn_act, which then skips its own statistics pass."""
    sums = None
    if want_bn_stats and _conv_precision != 0 and not out_lanes:
        sums = _stat_zeros(2 * weight.shape[0], x.device)
    out = _Conv2d.apply(x, weight, bias, int(stride), int(padding), int(dilation), int(out_lanes), sums)
    if sums is not None and getattr(sums, '_pxl_filled', False):
        out._pxl_bn_sums = sums
    return out


class _Aspp(torch.autograd.Function):
    """Classifier_Module.forward (deeplab_v2.py:81-85): sum of 4 dilated 3x3 convs (2048 -> C, with
    bias) as ONE 36-tap convolution that reads the latent once.  Output: channels_last
    [N, ldo=32, h, w] whose first C channels are the logits at latent resolution."""
    LDO = 32

    @staticmethod
    def forward(ctx, x, dilations, *wb):
        _chk(x, 'x', cl=True)
        nb = len(dilations)
        weights, biases = wb[:nb], wb[nb:]
        N, Cin, H, W = x.shape
        C = weights[0].shape[0]
        ldo = max(_Aspp.LDO, (C + 3) // 4 * 4)
        taps = []
        for d in dilations:
            taps += _taps(3, 3, d, d)
        # pack [ldo][9*nb][Cin]; rows >= C stay zero (they pad the dgrad operand)
        wp = torch.zeros((ldo, 9 * nb, Cin), dtype=torch.float32, device=x.device)
        for i, wgt in enumerate(weights):
            _chk(wgt, 'aspp weight', cl=True)
            wp[:C, 9 * i:9 * i + 9] = wgt.permute(0, 2, 3, 1).reshape(C, 9, Cin)
        bsum = biases[0]
        for b in biases[1:]:
            bsum = bsum + b
        out = conv_raw(x, wp, bsum.contiguous(), taps, N, H, W, Cin, H, W, C, ldo, 1, 1)
        ctx.save_for_backward(x, wp)
        ctx.meta = (taps, N, H, W, Cin, C, ldo, nb)
        return out

    @staticmethod
    def backward(ctx, dy):
        x, wp = ctx.saved_tensors
        taps, N, H, W, Cin, C, ldo, nb = ctx.meta
        dy = as_cl(dy)          # [N, ldo, H, W]; lanes >= C are zero (bilinear backward zero-fills)
        dx = None
        if ctx.needs_input_grad[0]:
            wt = transpose_weights(wp, ldo, 9 * nb, Cin)          # [Cin][36][ldo]
            dx = conv_raw(dy, wt, None, [-v for v in taps], N, H, W, ldo, H, W, Cin, Cin, 1, 1)
        dwp = torch.zeros((C, 9 * nb, Cin), dtype=torch.float32, device=dy.device)
        conv_wgrad_raw(x, dy, dwp, taps, N, H, W, Cin, H, W, C, ldo, 1, 1)
        db = torch.empty(C, dtype=torch.float32, device=dy.device)
        call('pxl_bias_grad', _p(dy), N * H * W, C, ldo, _p(db), 0, _stream())
        dws = [dwp[:, 9 * i:9 * i + 9].reshape(C, 3, 3, Cin).permute(0, 3, 1, 2) for i in range(nb)]
        return (dx, None) + tuple(dws) + tuple(db for _ in range(nb))


class _AsppGemm(torch.autograd.Function):
    """Classifier_Module.forward (deeplab_v2.py:81-85) on the fp16-pair tensor-core path: the channel contraction of
    all taps as ONE 1x1 GEMM (N = taps*C, the latent is read once), then a gather that adds the taps
    (csrc/aspp_gather.cu).  Backward: dZ = scatter(dY) as an fp16 pair, dX = dZ * W'^T and dW' = dZ^T * X are plain
    1x1 dgrad / wgrad GEMMs with K = taps*C and N = taps*C.  Same output layout as _Aspp."""
    LDO = 32

    @staticmethod
    def forward(ctx, x, dilations, *wb):
        nb = len(dilations)
        weights, biases = wb[:nb], wb[nb:]
        N, Cin, H, W = x.shape
        C = weights[0].shape[0]
        prec = _conv_precision
        want_lo = prec == 3
        ldo = max(_AsppGemm.LDO, (C + 3) // 4 * 4)
        taps = []
        for d in dilations:
            taps += _taps(3, 3, d, d)
        T = 9 * nb
        ldz = (T * C + 63) // 64 * 64                      # 36*21 = 756 -> 768
        # W' [ldz][Cin]: row t*C + co = W_t[co, :]
        wq = torch.zeros((ldz, Cin), dtype=torch.float32, device=x.device)
        for i, wgt in enumerate(weights):
            _chk(wgt, 'aspp weight', cl=True)
            wq[9 * i * C:9 * (i + 1) * C] = wgt.detach().permute(2, 3, 0, 1).reshape(9 * C, Cin)    # (kh,kw,co,ci)
        wh = h16_split(wq, H16_W_SCALE, want_lo)
        bsum = biases[0]
        for b in biases[1:]:
            bsum = bsum + b
        xh = _pair_of(x, want_lo)
        z = conv_raw(xh, wh, None, [0, 0], N, H, W, Cin, H, W, ldz, ldz, 1, 1, precision=prec)
        out = torch.empty((N, ldo, H, W), dtype=torch.float32, device=x.device, memory_format=CL)
        call('pxl_aspp_gather', _p(z), _p(bsum.detach().contiguous()), _p(out), N, H, W, C, ldz, ldo, _ctaps(taps), T, _stream())
        ctx.save_for_backward(xh.buf, wq)
        ctx.meta = (taps, N, H, W, Cin, C, ldo, ldz, nb, xh.scale, want_lo, prec)
        return out

    @staticmethod
    def backward(ctx, dy):
        xbuf, wq = ctx.saved_tensors
        taps, N, H, W, Cin, C, ldo, ldz, nb, xscale, want_lo, prec = ctx.meta
        dy = as_cl(dy)          # [N, ldo, H, W]; lanes >= C are zero (bilinear backward zero-fills)
        dev = dy.device
        T = 9 * nb
        n = N * H * W * ldz
        slot = _scale_slot(dev)
        call('pxl_h16_absmax', _p(dy), dy.numel(), _p(slot), _stream())
        dz = torch.empty((2, n), dtype=torch.float16, device=dev)
        call('pxl_aspp_scatter_h16', _p(dy), _p(dz[0]), _p(dz[1] if want_lo else None), _p(slot), H16_GRAD_TARGET_LOG2,
             N, H, W, C, ldo, ldz, _ctaps(taps), T, _stream())
        dzh = H16(dz, n, None, slot, want_lo)
        dx = None
        if ctx.needs_input_grad[0]:
            wt = h16_split(wq.t().contiguous(), H16_W_SCALE, want_lo)            # [Cin][ldz]
            dx = conv_raw(dzh, wt, None, [0, 0], N, H, W, ldz, H, W, Cin, Cin, 1, 1, precision=prec)
        dwq = torch.zeros((ldz, Cin), dtype=torch.float32, device=dev)
        conv_wgrad_raw(H16(xbuf, xbuf.shape[1], xscale, None, want_lo), dzh, dwq, [0, 0], N, H, W, Cin, H, W, ldz, ldz, 1, 1,
                       precision=prec)
        db = torch.empty(C, dtype=torch.float32, device=dev)
        call('pxl_bias_grad', _p(dy), N * H * W, C, ldo, _p(db), 0, _stream())
        g = dwq[:T * C].view(nb, 3, 3, C, Cin)                                   # (branch, kh, kw, co, ci)
        dws = [g[i].permute(2, 3, 0, 1) for i in range(nb)]                      # logical [C, Cin, 3, 3], CL strides
        return (dx, None) + tuple(dws) + tuple(db for _ in range(nb))


def aspp(x, weights, biases, dilations=(6, 12, 18, 24)):
    if _conv_precision >= 3 and x.shape[1] % 64 == 0:
        return _AsppGemm.apply(x, tuple(dilations), *(tuple(weights) + tuple(biases)))
    return _Aspp.apply(x, tuple(dilations), *(tuple(weights) + tuple(biases)))


class _Stem(torch.autograd.Function):
    """conv 7x7/2 pad 3 on the planar image -> NHWC (resnet.py:69,121); no input gradient.

    fp32 mode: the dedicated FFMA kernels.  Tensor-core modes: the image is unfolded once into a
    [pixels, 160] matrix (147 taps*channels + 13 zero lanes) and the stem runs as a flat 1x1 convolution on
    tcgen05, forward and wgrad sharing the matrix (19.9 GFLOP each on the 513x513 x16 batch)."""

    @staticmethod
    def forward(ctx, img, weight, sums):
        _chk(img, 'img'); _chk(weight, 'weight', cl=True)
        N, C, H, W = img.shape
        if C != 3 or tuple(weight.shape) != (64, 3, 7, 7):
            raise ValueError('stem expects a 3-channel image and a [64,3,7,7] weight')
        OH, OW = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
        out = torch.empty((N, 64, OH, OW), dtype=torch.float32, device=img.device, memory_format=CL)
        prec = _conv_precision
        ctx.meta = (N, H, W, OH, OW, prec)
        if prec == 0:
            call('pxl_stem_conv7x7s2', _p(img), _p(weight), _p(out), N, H, W, OH, OW, _stream())
            ctx.save_for_backward(img)
            return out
        if prec >= 3:
            # fp16-pair path: the unfolded matrix is written directly as the hi / lo planes [pixels][192]
            want_lo = prec == 3
            n = N * OH * OW * 192
            buf = torch.empty((2, n), dtype=torch.float16, device=img.device)
            call('pxl_stem_im2col_h16', _p(img), _p(buf[0]), _p(buf[1] if want_lo else None), float(H16_ACT_SCALE),
                 N, H, W, OH, OW, _stream())
            colsh = H16(buf, n, H16_ACT_SCALE, None, want_lo)
            wp = torch.zeros((64, 192), dtype=torch.float32, device=img.device)
            wp[:, :147] = weight.detach().permute(0, 2, 3, 1).reshape(64, 147)
            conv_raw(colsh, h16_split(wp, H16_W_SCALE, want_lo), None, [0, 0], N, OH, OW, 192, OH, OW, 64, 64, 1, 1, out=out,
                     precision=prec, bn_stats=sums)
            ctx.save_for_backward(buf if ctx.needs_input_grad[1] else None)
            ctx.h16 = want_lo
            return out
        cols = torch.empty((N, 160, OH, OW), dtype=torch.float32, device=img.device, memory_format=CL)
        call('pxl_stem_im2col', _p(img), _p(cols), N, H, W, OH, OW, _stream())
        wp = torch.zeros((64, 160), dtype=torch.float32, device=img.device)
        wp[:, :147] = weight.detach().permute(0, 2, 3, 1).reshape(64, 147)      # physical order of the CL weight
        conv_raw(cols, wp, None, [0, 0], N, OH, OW, 160, OH, OW, 64, 64, 1, 1, out=out, precision=prec, bn_stats=sums)
        ctx.save_for_backward(cols if ctx.needs_input_grad[1] else None)
        return out

    @staticmethod
    def backward(ctx, dy):
        (saved,) = ctx.saved_tensors
        N, H, W, OH, OW, prec = ctx.meta
        dy = as_cl(dy)
        if prec == 0:
            dw = torch.empty((64, 3, 7, 7), dtype=torch.float32, device=dy.device, memory_format=CL).zero_()
            call('pxl_stem_conv7x7s2_wgrad', _p(saved), _p(dy), _p(dw), N, H, W, OH, OW, _stream())
            return None, dw, None
        if prec >= 3:
            dwp = torch.zeros((64, 192), dtype=torch.float32, device=dy.device)
            conv_wgrad_raw(H16(saved, saved.shape[1], H16_ACT_SCALE, None, ctx.h16), dy, dwp, [0, 0], N, OH, OW, 192, OH, OW, 64, 64,
                           1, 1, precision=prec)
            dw = dwp[:, :147].reshape(64, 7, 7, 3).permute(0, 3, 1, 2)
            return None, dw, None
        dwp = torch.zeros((64, 160), dtype=torch.float32, device=dy.device)
        conv_wgrad_raw(saved, dy, dwp, [0, 0], N, OH, OW, 160, OH, OW, 64, 64, 1, 1, precision=prec)
        dw = dwp[:, :147].reshape(64, 7, 7, 3).permute(0, 3, 1, 2)              # logical [64,3,7,7], CL strides
        return None, dw, None


def stem_conv(img, weight, want_bn_stats=False):
    """want_bn_stats: like conv2d - on the tensor-core path the epilogue accumulates the BN sums."""
    sums = _stat_zeros(128, img.device) if (want_bn_stats and _conv_precision != 0) else None
    out = _Stem.apply(img.contiguous(), weight, sums)
    if sums is not None and getattr(sums, '_pxl_filled', False):
        out._pxl_bn_sums = sums
    return out


# ------------------------------------------------------------------------------------------------
# batch norm (+ReLU, +residual), max-pool
# ------------------------------------------------------------------------------------------------

# process group (by id) -> nn.peer.PeerExchange; registered by EngineParallel when CUDA IPC is available
_peer_exchanges = {}


def register_peer_exchange(group, exchange):
    if exchange is None:
        _peer_exchanges.pop(id(group), None)
    else:
        _peer_exchanges[id(group)] = exchange


class _BnAct(torch.autograd.Function):
    """_SynchronizedBatchNorm.forward (batchnorm.py:48-78) fused with the ReLU / residual add that
    follow it in Bottleneck.forward (resnet.py:33-48).  ``group``: torch.distributed group whose
    ranks share batch statistics (the reference's cross-replica SyncBN); None = local."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, residual, training, momentum, eps, relu, group, clamp_var, sums=None):
        _chk(x, 'x', cl=True)
        N, C, H, W = x.shape
        rows = N * H * W
        dev = x.device
        y = torch.empty_like(x)
        coeff = torch.empty((4, C), dtype=torch.float32, device=dev)     # mean, invstd, scale, shift
        count = float(rows)
        clamp = 1 if clamp_var else 0
        applied = False
        if training:
            if sums is None:
                sums = _stat_zeros(2 * C, dev)
                call('pxl_bn_stats', _p(x), rows, C, _p(sums), _stream())
            fused = False
            if group is not None:
                import torch.distributed as dist
                count = float(rows) * dist.get_world_size(group)
                clamp = 1     # batchnorm.py:125: the multi-replica path clamps var instead of adding eps
                px = _peer_exchanges.get(id(group))
                if px is not None and 2 * C <= 4096:
                    # NVLink peer-memory exchange fused with the finalize (csrc/peer_exchange.cu)
                    px.allreduce_bn(sums, (count, C, gamma, beta, running_mean, running_var, momentum, eps, clamp,
                                           coeff[0], coeff[1], coeff[2], coeff[3]))
                    fused = True
                else:
                    dist.all_reduce(sums, group=group)
            if residual is not None:
                _chk(residual, 'residual', cl=True)
            if group is None and FUSE_BN_FINALIZE:
                # local statistics: finalize + apply in one launch
                call('pxl_bn_finalize_apply', _p(x), _p(sums), count, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
                     float(momentum), float(eps), clamp, _p(coeff[0]), _p(coeff[1]), _p(coeff[2]), _p(coeff[3]),
                     _p(residual), int(relu), _p(y), rows, C, _stream())
                applied = True
            elif not fused:
                call('pxl_bn_finalize', _p(sums), count, C, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
                     float(momentum), float(eps), clamp, _p(coeff[0]), _p(coeff[1]), _p(coeff[2]), _p(coeff[3]), _stream())
        else:
            call('pxl_bn_eval_coeffs', C, _p(gamma), _p(beta), _p(running_mean), _p(running_var), float(eps),
                 _p(coeff[2]), _p(coeff[3]), _stream())
            if torch.is_grad_enabled() and (x.requires_grad or gamma.requires_grad):
                # eval-mode BN inside a training graph (freeze_bn): the backward treats the running statistics as
                # constants; mean / inv_std slots hold them for bn_bwd_reduce (tiny per-channel torch ops)
                coeff[0].copy_(running_mean)
                coeff[1].copy_(torch.rsqrt(running_var + eps))
        if not applied:
            if residual is not None:
                _chk(residual, 'residual', cl=True)
            call('pxl_bn_apply', _p(x), _p(coeff[2]), _p(coeff[3]), _p(residual), int(relu), _p(y), rows, C, _stream())
        ctx.save_for_backward(x, y if (relu and residual is not None) else None, gamma, coeff, running_var, beta)
        ctx.meta = (rows, C, count, bool(relu), residual is not None, bool(training), float(eps), group)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, gamma, coeff, running_var, beta = ctx.saved_tensors
        rows, C, count, relu, has_res, training, eps, group = ctx.meta
        dy = as_cl(dy)
        dev = dy.device
        dsums = _stat_zeros(2 * C, dev)
        if not training:
            # F.batch_norm(training=False) backward: dx = dz * gamma / sqrt(running_var + eps), d(gamma) = sum dz * xhat,
            # d(beta) = sum dz with xhat from the running statistics.  The reduce launch gives the parameter sums; the
            # dx launch runs with zero batch sums, which removes its mean terms.
            ymask = y if (relu and has_res) else None
            call('pxl_bn_bwd_reduce', _p(x), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), int(relu), rows, C, _p(dsums),
                 _p(coeff[2]), _p(coeff[3]), _stream())
            dgamma = torch.empty(C, dtype=torch.float32, device=dev)
            dbeta = torch.empty(C, dtype=torch.float32, device=dev)
            call('pxl_bn_bwd_params', _p(dsums), C, _p(dgamma), _p(dbeta), 0, _stream())
            zsums = _stat_zeros(2 * C, dev)
            dx = torch.empty_like(x)
            dres = torch.empty_like(x) if has_res else None
            call('pxl_bn_bwd_dx', _p(x), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), _p(gamma), _p(zsums), count, int(relu),
                 _p(dx), _p(dres), rows, C, _p(coeff[2]), _p(coeff[3]), _p(None), _p(None), _stream())
            return dx, dgamma, dbeta, None, None, dres, None, None, None, None, None, None, None
        # ReLU without residual: the mask is recomputed from x (same fmaf as the forward) instead of reading y
        ymask = y if (relu and has_res) else None
        call('pxl_bn_bwd_reduce', _p(x), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), int(relu), rows, C, _p(dsums),
             _p(coeff[2]), _p(coeff[3]), _stream())
        # single GPU with arena gradients in place: the dx launch adds d(gamma), d(beta) straight into .grad
        grads_in_arena = (ACCUM_WGRAD_INPLACE and gamma.grad is not None and beta.grad is not None
                          and gamma.grad.is_contiguous() and beta.grad.is_contiguous())
        px = _peer_exchanges.get(id(group)) if group is not None else None
        if px is not None and 2 * C > 4096:
            px = None
        # d(gamma), d(beta) come from the LOCAL sums (DDP averages them with the other gradients); whenever the
        # gradient arena is in place they are accumulated by a launch that runs anyway: the dx kernel (single GPU)
        # or the peer-exchange kernel (before it exchanges the sums)
        acc_inplace = grads_in_arena and group is None
        acc_in_exchange = grads_in_arena and px is not None
        dgamma = dbeta = None
        if not (acc_inplace or acc_in_exchange):
            dgamma = torch.empty(C, dtype=torch.float32, device=dev)
            dbeta = torch.empty(C, dtype=torch.float32, device=dev)
            call('pxl_bn_bwd_params', _p(dsums), C, _p(dgamma), _p(dbeta), 0, _stream())
        if group is not None:
            if px is not None:
                px.allreduce_bn(dsums, param_grads=(gamma.grad, beta.grad) if acc_in_exchange else None)
            else:
                import torch.distributed as dist
                dist.all_reduce(dsums, group=group)
        dx = torch.empty_like(x)
        dres = torch.empty_like(x) if has_res else None
        call('pxl_bn_bwd_dx', _p(x), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), _p(gamma), _p(dsums), count, int(relu),
             _p(dx), _p(dres), rows, C, _p(coeff[2]), _p(coeff[3]),
             _p(gamma.grad if acc_inplace else None), _p(beta.grad if acc_inplace else None), _stream())
        return dx, dgamma, dbeta, None, None, dres, None, None, None, None, None, None, None


def bn_act(x, gamma, beta, running_mean, running_var, training=True, momentum=0.1, eps=1e-5, relu=False,
           residual=None, group=None, clamp_var=False):
    """clamp_var: use the reference's multi-replica formula inv_std = clamp(var, eps)^-1/2
    (batchnorm.py:125) instead of (var + eps)^-1/2; implied when ``group`` spans several ranks."""
    sums = getattr(x, '_pxl_bn_sums', None) if training else None      # produced by the conv epilogue
    return _BnAct.apply(x, gamma, beta, running_mean, running_var, residual, bool(training), float(momentum),
                        float(eps), bool(relu), group, bool(clamp_var), sums)


# ------------------------------------------------------------------------------------------------
# conv -> BN -> (+residual) -> (ReLU) as one node on the fp16-pair path
# ------------------------------------------------------------------------------------------------

# Weight gradients are off the critical path of the backward pass (nothing reads them before the optimiser step), so
# they could run on a side stream right after the dX pair they consume exists, overlapping the HBM-bound BatchNorm
# backward launches.  NEGATIVE RESULT (measured, B200, MT step): 53.8 ms -> 76.4 ms.  The wgrad CTAs (200 KB of
# shared memory each) take SMs away from the persistent one-CTA-per-SM convolutions of the critical path, which then
# wait for them - a priority inversion the default stream cannot be prioritised out of.  Opt-in: PXL_WGRAD_SIDE_STREAM=1.
# block outputs: ReLU mask for the backward as 1 byte per 4 values (A/B switch; 0 re-reads the fp32 result)
BN_RELU_MASK = _os.environ.get('PXL_BN_RELU_MASK', '1') != '0'
WGRAD_SIDE_STREAM = _os.environ.get('PXL_WGRAD_SIDE_STREAM', '0') != '0'
_side_streams = {}


def _wgrad_stream(device):
    s = _side_streams.get(device)
    if s is None:
        s = _side_streams[device] = [torch.cuda.Stream(device=device), False, False]
    return s


def _join_after_backward():
    for ent in _side_streams.values():
        ent[2] = False
    join_side_streams()


def join_side_streams():
    """Make the current stream wait for every side-stream launch so far (called before gradients are consumed:
    all-reduce, optimiser step, zero_grad)."""
    for ent in _side_streams.values():
        if ent[1]:
            torch.cuda.current_stream().wait_stream(ent[0])
            ent[1] = False


_residual_stash = {}            # block key -> gradient of the residual branch waiting for the block's first dgrad (one step)
H16_DX_TARGET_LOG2 = 12         # bn_bwd_dx: max|gamma*invstd| * absmax(dz) -> <= 2^12, 3 bits of headroom for the mean terms
_unit_out_pair = None           # H16 of the last _ConvBnAct.forward output (picked up by conv_bn_act right after apply)


def _pair_of(x, want_lo):
    """The fp16 pair of an activation: attached by its producer (same step, unmodified), else split now (cached)."""
    ent = getattr(x, '_pxl_h16', None)
    if ent is not None and ent[0] == _epoch and ent[1] == x._version and ent[2] == x.data_ptr() and ent[3].has_lo >= want_lo:
        return ent[3]
    if getattr(x, '_pxl_carrier', False):
        raise RuntimeError('fp16-pair carrier tensor without a valid pair (stale step?)')
    return h16_cached(x, H16_ACT_SCALE, want_lo)


def _attach_pair(t, h, carrier=False):
    t._pxl_h16 = (_epoch, t._version, t.data_ptr(), h)
    if carrier:
        t._pxl_carrier = True
    return t


def is_carrier(t):
    """True for tensors whose storage holds an fp16 pair instead of fp32 values (inner activations of a bottleneck
    on the fp16-pair path): only pair-aware consumers (conv_bn_act) may read them."""
    return getattr(t, '_pxl_carrier', False)


class _ConvBnAct(torch.autograd.Function):
    """Bottleneck building block (resnet.py:33-48): bias-free conv -> train-mode (Sync)BN (batchnorm.py:48-78)
    -> (+ residual) -> (ReLU), ONE autograd node on the kind::f16 tensor-core path.

    Forward: the convolution reads the fp16 pair of its input, its epilogue produces the BN statistics, and the BN
    apply launch writes its result directly as the fp16 pair of the next convolution (``out_mode`` 'pair': only the
    pair, carried by a float32-typed tensor over the same storage; 'both': fp32 tensor + attached pair; 'fp32').
    Backward: the BN dx launch writes dX of the convolution output as an fp16 pair with a device-side power-of-two
    scale; dgrad and wgrad read it.  No fp16 pair ever takes an extra trip through HBM, and gradients between nodes
    stay fp32."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, running_mean, running_var, residual, stride, padding, dilation,
                momentum, eps, relu, group, clamp_var, out_mode, stash_key=None, stash_role=None):
        global _unit_out_pair
        ctx.stash = (stash_key, stash_role)
        prec = _conv_precision
        want_lo = prec == 3
        N, Cin, H, W = x.shape
        Cout, Cin2, kh, kw = weight.shape
        if Cin2 != Cin:
            raise ValueError('channel mismatch')
        OH = (H + 2 * padding - dilation * (kh - 1) - 1) // stride + 1
        OW = (W + 2 * padding - dilation * (kw - 1) - 1) // stride + 1
        taps = _taps(kh, kw, dilation, padding)
        xh = _pair_of(x, want_lo)
        dev = xh.device
        sums = _stat_zeros(2 * Cout, dev)
        c = conv_raw(xh, weight, None, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1, bn_stats=sums)
        rows = N * OH * OW
        n = rows * Cout
        count = float(rows)
        clamp = 1 if clamp_var else 0
        coeff = torch.empty((4, Cout), dtype=torch.float32, device=dev)
        pair = torch.empty((2, n), dtype=torch.float16, device=dev) if out_mode != 'fp32' else None
        y = torch.empty_like(c) if out_mode != 'pair' else None
        hi = pair[0] if pair is not None else None
        lo = pair[1] if (pair is not None and want_lo) else None
        # block output (residual + ReLU): the backward takes the ReLU mask from one byte per 4 values instead of
        # re-reading the fp32 result in both of its launches
        mask = (torch.empty(n // 4, dtype=torch.uint8, device=dev)
                if (BN_RELU_MASK and relu and residual is not None and any(ctx.needs_input_grad)) else None)
        if residual is not None:
            _chk(residual, 'residual', cl=True)
        applied = fused = False
        if group is not None:
            import torch.distributed as dist
            count = float(rows) * dist.get_world_size(group)
            clamp = 1     # batchnorm.py:125: the multi-replica path clamps var instead of adding eps
            px = _peer_exchanges.get(id(group))
            if px is not None and 2 * Cout <= 4096:
                px.allreduce_bn(sums, (count, Cout, gamma, beta, running_mean, running_var, momentum, eps, clamp,
                                       coeff[0], coeff[1], coeff[2], coeff[3]))
                fused = True
            else:
                dist.all_reduce(sums, group=group)
        if group is None and FUSE_BN_FINALIZE:
            call('pxl_bn_finalize_apply_h16', _p(c), _p(sums), count, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
                 float(momentum), float(eps), clamp, _p(coeff[0]), _p(coeff[1]), _p(coeff[2]), _p(coeff[3]),
                 _p(residual), int(relu), _p(y), rows, Cout, _p(hi), _p(lo), float(H16_ACT_SCALE), _p(mask), _stream())
            applied = True
        elif not fused:
            call('pxl_bn_finalize', _p(sums), count, Cout, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
                 float(momentum), float(eps), clamp, _p(coeff[0]), _p(coeff[1]), _p(coeff[2]), _p(coeff[3]), _stream())
        if not applied:
            call('pxl_bn_apply_h16', _p(c), _p(coeff[2]), _p(coeff[3]), _p(residual), int(relu), _p(y), rows, Cout,
                 _p(hi), _p(lo), float(H16_ACT_SCALE), _p(mask), _stream())
        ctx.save_for_backward(xh.buf, weight, c, mask if BN_RELU_MASK else (y if (relu and residual is not None) else None),
                              gamma, coeff, beta)
        ctx.meta = (taps, N, H, W, Cin, OH, OW, Cout, stride, kh * kw, count, bool(relu), residual is not None, group,
                    xh.scale, want_lo, prec)
        _unit_out_pair = H16(pair, n, H16_ACT_SCALE, None, want_lo) if pair is not None else None
        if out_mode == 'pair':
            return pair.view(torch.float32).view(N, OH, OW, Cout).permute(0, 3, 1, 2)
        return y

    @staticmethod
    def backward(ctx, dy):
        xbuf, weight, c, mask, gamma, coeff, beta = ctx.saved_tensors
        taps, N, H, W, Cin, OH, OW, Cout, stride, T, count, relu, has_res, group, xscale, want_lo, prec = ctx.meta
        if is_carrier(dy):
            raise RuntimeError('gradient tensors are never fp16-pair carriers')
        dy = as_cl(dy)
        dev = dy.device
        rows = N * OH * OW
        n = rows * Cout
        C = Cout
        dsums = _stat_zeros(2 * C, dev)
        slot = _scale_slot(dev)
        if relu and has_res and mask is None:
            raise RuntimeError('the ReLU mask of a residual unit was not recorded in the forward')
        ymask = None
        if mask is not None and mask.dtype != torch.uint8:      # PXL_BN_RELU_MASK=0: the fp32 result is the mask
            ymask, mask = mask, None
        call('pxl_bn_bwd_reduce_h16', _p(c), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), int(relu), rows, C, _p(dsums),
             _p(coeff[2]), _p(coeff[3]), _p(slot), _p(mask), _stream())
        grads_in_arena = (ACCUM_WGRAD_INPLACE and gamma.grad is not None and beta.grad is not None
                          and gamma.grad.is_contiguous() and beta.grad.is_contiguous())
        px = _peer_exchanges.get(id(group)) if group is not None else None
        if px is not None and 2 * C > 4096:
            px = None
        acc_inplace = grads_in_arena and group is None
        acc_in_exchange = grads_in_arena and px is not None
        dgamma = dbeta = None
        if not (acc_inplace or acc_in_exchange):
            dgamma = torch.empty(C, dtype=torch.float32, device=dev)
            dbeta = torch.empty(C, dtype=torch.float32, device=dev)
            call('pxl_bn_bwd_params', _p(dsums), C, _p(dgamma), _p(dbeta), 0, _stream())
        if group is not None:
            if px is not None:
                px.allreduce_bn(dsums, param_grads=(gamma.grad, beta.grad) if acc_in_exchange else None)
            else:
                import torch.distributed as dist
                dist.all_reduce(dsums, group=group)
        dpair = torch.empty((2, n), dtype=torch.float16, device=dev)
        dres = torch.empty_like(c) if has_res else None
        call('pxl_bn_bwd_dx_h16', _p(c), _p(ymask), _p(dy), _p(coeff[0]), _p(coeff[1]), _p(gamma), _p(dsums), count, int(relu),
             _p(None), _p(dres), rows, C, _p(coeff[2]), _p(coeff[3]),
             _p(gamma.grad if acc_inplace else None), _p(beta.grad if acc_inplace else None),
             _p(dpair[0]), _p(dpair[1] if want_lo else None), _p(slot), H16_DX_TARGET_LOG2, _p(mask), _stream())
        dh = H16(dpair, n, None, slot, want_lo)
        dx = dw = None
        stash_key, stash_role = ctx.stash
        if stash_role == 'give' and dres is not None:
            # the residual branch of this block is the block input itself: its gradient is handed to the block's first
            # unit, whose dgrad epilogue adds into it (TMA reduce-add) - no elementwise add of the two branch gradients
            _residual_stash[stash_key] = dres
            dres = None
        give_dx = stash_role == 'give_dx' and _residual_stash.get(stash_key) is None
        if ctx.needs_input_grad[0]:
            arena, off = _arena_of(weight) if BATCH_WEIGHT_PREP else (None, None)
            if arena is not None and arena._conv_at.get(off) == (Cout, T, Cin):
                nw = weight.numel()
                wt = H16(arena.derived('h16_t')[:, off:off + nw], nw, H16_W_SCALE, None, True)
            else:
                wt = h16_split(transpose_weights(weight, Cout, T, Cin), H16_W_SCALE, want_lo)
            held = _residual_stash.pop(stash_key, None) if stash_role == 'take' else None
            if stash_role == 'take' and held is None:
                _residual_stash[stash_key] = 'taken'          # a 'give_dx' unit that runs later returns its dX itself
            if held is not None:
                try:
                    dx = conv_raw(dh, wt, None, [-v for v in taps], N, OH, OW, Cout, H, W, Cin, Cin, 1, stride, out=held,
                                  precision=prec, accumulate=True)
                except _lib.PxlError as e:
                    if e.code != _lib.PXL_ERR_UNSUPPORTED:
                        raise
                    dx = conv_raw(dh, wt, None, [-v for v in taps], N, OH, OW, Cout, H, W, Cin, Cin, 1, stride, precision=prec)
                    dx += held
            else:
                dx = conv_raw(dh, wt, None, [-v for v in taps], N, OH, OW, Cout, H, W, Cin, Cin, 1, stride, precision=prec)
        elif stash_role == 'take':
            _residual_stash.pop(stash_key, None)
        if give_dx and dx is not None:
            # downsample unit of a bottleneck: the block input also feeds conv1, whose backward runs later (autograd
            # executes later-created nodes first; conv1 waits for conv2's backward) and adds its dX into this buffer
            _residual_stash[stash_key] = dx
            dx = None
        if ctx.needs_input_grad[1]:
            inplace = ACCUM_WGRAD_INPLACE and weight.grad is not None and weight.grad.is_contiguous(memory_format=CL)
            dwbuf = weight.grad if inplace else torch.zeros_like(weight, memory_format=torch.preserve_format)
            xh = H16(xbuf, xbuf.shape[1], xscale, None, want_lo)
            if WGRAD_SIDE_STREAM and inplace:
                ent = _wgrad_stream(dev)
                main = torch.cuda.current_stream()
                ev = torch.cuda.Event()
                ev.record(main)                         # the dX pair (and everything before it) is enqueued
                ent[0].wait_event(ev)
                with torch.cuda.stream(ent[0]):
                    conv_wgrad_raw(xh, dh, dwbuf, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1, precision=prec)
                dpair.record_stream(ent[0])
                xbuf.record_stream(ent[0])
                ent[1] = True
                if not ent[2]:
                    # whoever reads .grad after loss.backward() does so on the main stream: join when this backward ends
                    ent[2] = True
                    torch.autograd.Variable._execution_engine.queue_callback(_join_after_backward)
            else:
                conv_wgrad_raw(xh, dh, dwbuf, taps, N, H, W, Cin, OH, OW, Cout, Cout, stride, 1, precision=prec)
            dw = None if inplace else dwbuf
        return (dx, dw, dgamma, dbeta, None, None, dres) + (None,) * 11


def conv_bn_unit_ok(conv, bn):
    """True when conv -> bn can run as one _ConvBnAct node: fp16-pair precision, train-mode BN, bias-free conv with
    64-aligned channel counts and stride 1 / 2."""
    return (_conv_precision >= 3 and bn.training and conv.bias is None and not conv.out_lanes
            and conv.in_channels % 64 == 0 and conv.out_channels % 64 == 0 and conv.stride in (1, 2))


def conv_bn_act(x, conv, bn, relu=False, residual=None, out_mode='both', stash_key=None, stash_role=None):
    """conv (nn.modules.Conv2d) -> bn (nn.modules.BatchNorm2d) -> (+residual) -> (ReLU); see _ConvBnAct.
    stash_key / stash_role: a bottleneck whose residual branch is its own input marks its last unit 'give' and its
    first unit 'take' with a common key - the residual gradient then reaches the block input through the first
    unit's dgrad epilogue (out += ...) instead of through autograd's add."""
    global _unit_out_pair
    if not is_carrier(x):
        x = as_cl(x)
    out = _ConvBnAct.apply(x, conv.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, residual,
                           int(conv.stride), int(conv.padding), int(conv.dilation), float(bn.momentum), float(bn.eps),
                           bool(relu), bn.sync_group, bool(bn.multi_replica_formula), out_mode, stash_key, stash_role)
    pair, _unit_out_pair = _unit_out_pair, None
    if pair is not None:
        _attach_pair(out, pair, carrier=(out_mode == 'pair'))
    return out


class _MaxPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _chk(x, 'x', cl=True)
        N, C, H, W = x.shape
        OH, OW = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
        y = torch.empty((N, C, OH, OW), dtype=torch.float32, device=x.device, memory_format=CL)
        call('pxl_maxpool3x3s2_fwd', _p(x), _p(y), N, H, W, C, OH, OW, _stream())
        ctx.save_for_backward(x)
        ctx.meta = (N, H, W, C, OH, OW)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        N, H, W, C, OH, OW = ctx.meta
        dy = as_cl(dy)
        dx = torch.empty_like(x)
        call('pxl_maxpool3x3s2_bwd', _p(x), _p(None), _p(dy), _p(dx), N, H, W, C, OH, OW, _stream())
        return dx


def maxpool3x3s2(x):
    """nn.MaxPool2d(kernel_size=3, stride=2, padding=1) on NHWC (resnet.py:72)."""
    return _MaxPool.apply(x)


# ------------------------------------------------------------------------------------------------
# optimiser / EMA on flat arenas
# ------------------------------------------------------------------------------------------------

def sgd_ema_(p, g, buf, teacher, lr, momentum, weight_decay, ema_d, first_step):
    call('pxl_sgd_ema', _p(p), _p(g), _p(buf), _p(teacher), p.numel(), float(lr), float(momentum),
         float(weight_decay), float(ema_d), int(first_step), _stream())


def ema_(teacher, student, ema_d):
    call('pxl_ema', _p(teacher), _p(student), teacher.numel(), float(ema_d), _stream())


def launch_count():
    return int(_lib.load().pxl_launch_count())


def reset_launch_count():
    _lib.load().pxl_reset_launch_count()


# ------------------------------------------------------------------------------------------------
# AdvSSL / GCT / CCT tails
# ------------------------------------------------------------------------------------------------

class _PlanarToNhwc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ldc, coff, out):
        _chk(x, 'x')
        n, c, h, w = x.shape
        if out is None:
            out = torch.empty((n, ldc, h, w), dtype=torch.float32, device=x.device, memory_format=CL)
            if ldc != c:
                out.zero_()
        call('pxl_planar_to_nhwc', _p(x), _p(out), n, c, h * w, ldc, coff, _stream())
        ctx.meta = (n, c, h, w, ldc, coff)
        return out

    @staticmethod
    def backward(ctx, g):
        n, c, h, w, ldc, coff = ctx.meta
        g = as_cl(g)
        dx = torch.empty((n, c, h, w), dtype=torch.float32, device=g.device)
        call('pxl_nhwc_to_planar', _p(g), _p(dx), n, c, h * w, ldc, coff, _stream())
        return dx, None, None, None


def planar_to_nhwc(x, ldc=None, coff=0):
    """planar [n,C,H,W] -> channels_last [n,ldc,H,W] with the C channels in lanes [coff, coff+C) and
    zeros elsewhere (the conv input of FCDiscriminator / FlawDetector)."""
    c = x.shape[1]
    if ldc is None:
        ldc = (c + 31) // 32 * 32
    return _PlanarToNhwc.apply(x.contiguous(), int(ldc), int(coff), None)


class _CatPlanarToNhwc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ldc, *tensors):
        n, _, h, w = tensors[0].shape
        out = torch.empty((n, ldc, h, w), dtype=torch.float32, device=tensors[0].device, memory_format=CL)
        chans = [t.shape[1] for t in tensors]
        if sum(chans) != ldc:
            out.zero_()
        off = 0
        for t in tensors:
            _chk(t, 'cat input')
            call('pxl_planar_to_nhwc', _p(t), _p(out), n, t.shape[1], h * w, ldc, off, _stream())
            off += t.shape[1]
        ctx.meta = (n, h, w, ldc, chans)
        return out

    @staticmethod
    def backward(ctx, g):
        n, h, w, ldc, chans = ctx.meta
        g = as_cl(g)
        grads, off = [], 0
        for i, c in enumerate(chans):
            if ctx.needs_input_grad[1 + i]:
                dx = torch.empty((n, c, h, w), dtype=torch.float32, device=g.device)
                call('pxl_nhwc_to_planar', _p(g), _p(dx), n, c, h * w, ldc, off, _stream())
                grads.append(dx)
            else:
                grads.append(None)
            off += c
        return (None,) + tuple(grads)


def cat_planar_to_nhwc(tensors, ldc=None):
    """torch.cat(tensors, dim=1) of planar maps written straight into one zero-padded NHWC tensor
    (FlawDetector.forward, ssl_gct.py:566-567)."""
    ctot = sum(t.shape[1] for t in tensors)
    if ldc is None:
        ldc = (ctot + 31) // 32 * 32
    return _CatPlanarToNhwc.apply(int(ldc), *[t.contiguous() for t in tensors])


class _NhwcToPlanar(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, C):
        _chk(x, 'x', cl=True)
        n, ldc, h, w = x.shape
        out = torch.empty((n, C, h, w), dtype=torch.float32, device=x.device)
        call('pxl_nhwc_to_planar', _p(x), _p(out), n, C, h * w, ldc, 0, _stream())
        ctx.meta = (n, C, h, w, ldc)
        return out

    @staticmethod
    def backward(ctx, g):
        n, C, h, w, ldc = ctx.meta
        g = g.contiguous()
        dx = torch.empty((n, ldc, h, w), dtype=torch.float32, device=g.device, memory_format=CL)
        if ldc != C:
            dx.zero_()
        call('pxl_planar_to_nhwc', _p(g), _p(dx), n, C, h * w, ldc, 0, _stream())
        return dx, None


def nhwc_to_planar(x, channels):
    """First ``channels`` lanes of a channels_last tensor as a planar [n,channels,H,W] tensor."""
    return _NhwcToPlanar.apply(as_cl(x), int(channels))


def onehot_nhwc(labels, num_classes, ldc=None):
    """One-hot of float labels [n,1,H,W] as channels_last [n,ldc,H,W]; ignore pixels are all-zero."""
    _chk(labels, 'labels')
    n, _, h, w = labels.shape
    if ldc is None:
        ldc = (num_classes + 31) // 32 * 32
    out = torch.empty((n, ldc, h, w), dtype=torch.float32, device=labels.device, memory_format=CL).zero_()
    call('pxl_onehot_nhwc', _p(labels), _p(out), n * h * w, num_classes, ldc, 0, _stream())
    return out


class _LeakyRelu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, slope):
        y = torch.empty_like(x)
        call('pxl_leaky_relu_fwd', _p(x), _p(y), x.numel(), float(slope), _stream())
        ctx.save_for_backward(y)
        ctx.slope = float(slope)
        return y

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        g = g.contiguous(memory_format=CL) if y.is_contiguous(memory_format=CL) and y.dim() == 4 else g.contiguous()
        dx = torch.empty_like(y)
        call('pxl_leaky_relu_bwd', _p(y), _p(g), _p(dx), y.numel(), ctx.slope, _stream())
        return dx, None


def leaky_relu(x, slope=0.2):
    """nn.LeakyReLU(slope) (slope 0 = ReLU); x.numel() % 4 == 0."""
    return _LeakyRelu.apply(x, slope)


class _BceMasked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, labels, target, ignore_index):
        _chk(pred, 'pred')
        n = pred.shape[0]
        hw = pred.numel() // n
        per = torch.empty(n, dtype=torch.float32, device=pred.device)
        call('pxl_bce_logits_masked', _p(pred), _p(labels), float(target), int(ignore_index), n, hw, _p(per), _p(None),
             _p(None), 0.0, _stream())
        ctx.save_for_backward(pred, labels)
        ctx.meta = (float(target), int(ignore_index), n, hw)
        return per

    @staticmethod
    def backward(ctx, g):
        pred, labels = ctx.saved_tensors
        target, ignore, n, hw = ctx.meta
        per = torch.empty(n, dtype=torch.float32, device=pred.device)
        grad = torch.empty_like(pred)
        g = g.contiguous().float()
        call('pxl_bce_logits_masked', _p(pred), _p(labels), target, ignore, n, hw, _p(per), _p(grad), _p(g), 0.0, _stream())
        return grad, None, None, None


def bce_logits_masked(pred, labels, target, ignore_index=255):
    """FCDiscriminatorCriterion(ssladv_preprocess_fcd_criterion(pred, labels, is_real=target))
    -> per-sample loss [n] (ssl_adv.py:496-503 + task/sseg/func.py:137-155).  labels may be None."""
    if labels is not None:
        labels = labels.contiguous()
    return _BceMasked.apply(pred.contiguous(), labels, float(target), int(ignore_index))


def adam_(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step):
    call('pxl_adam', _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
         float(weight_decay), int(step), _stream())


_blur_weights = {}


def gaussian_kernel_1d(k, device):
    """1-D factor v of GaussianBlurLayer's k x k kernel (= outer(v, v)): scipy's gaussian_filter1d of a
    delta with sigma = 0.3*((k-1)/2 - 1) + 0.8, truncate 4 sigma, 'reflect' boundary
    (nn/module/gaussian_blur.py:52-64), evaluated here in closed form."""
    key = (k, str(device))
    if key not in _blur_weights:
        import math
        sigma = 0.3 * ((k - 1) * 0.5 - 1) + 0.8
        radius = int(4.0 * sigma + 0.5)
        xs = range(-radius, radius + 1)
        phi = [math.exp(-0.5 / (sigma * sigma) * x * x) for x in xs]
        tot = sum(phi)
        phi = [p / tot for p in phi]
        # correlate a delta at k//2 of a length-k signal with 'reflect' (d c b a | a b c d | d c b a) padding
        c = k // 2
        v = [0.0] * k
        for i in range(k):
            acc = 0.0
            for j, wgt in zip(xs, phi):
                pos = i + j
                # scipy 'reflect': mirror about the edge sample boundary (half-sample symmetric)
                while pos < 0 or pos >= k:
                    pos = -pos - 1 if pos < 0 else 2 * k - 1 - pos
                if pos == c:
                    acc += wgt
            v[i] = acc
        _blur_weights[key] = torch.tensor(v, dtype=torch.float64).to(torch.float32).to(device)
    return _blur_weights[key]


def gaussian_blur(x, k, clamp_min=None):
    """GaussianBlurLayer(1, k) on [n,1,H,W] maps (no autograd: the reference only blurs detached maps)."""
    _chk(x, 'x')
    n, c, h, w = x.shape
    if c != 1:
        raise ValueError('gaussian_blur expects single-channel maps')
    tmp, out = torch.empty_like(x), torch.empty_like(x)
    call('pxl_gauss_blur_sep', _p(x), _p(tmp), _p(out), n, h, w, int(k), _p(gaussian_kernel_1d(k, x.device)),
         float(-3.0e38 if clamp_min is None else clamp_min), _stream())
    return out


def dilate3x3_reflect(x):
    _chk(x, 'x')
    n, c, h, w = x.shape
    out = torch.empty_like(x)
    call('pxl_dilate3x3_reflect', _p(x), _p(out), n * c, h, w, _stream())
    return out


def minmax_norm(x, eps=1e-9, zero_below=-1.0):
    _chk(x, 'x')
    n = x.shape[0]
    out = torch.empty_like(x)
    call('pxl_minmax_norm', _p(x), _p(out), n, x.numel() // n, float(eps), float(zero_below), -3.0e38, _stream())
    return out


class _IBNorm(torch.autograd.Function):
    """IBNorm (ssl_gct.py:588-607): the first ``nb`` channels go through (Sync)BatchNorm (affine, running
    stats), the rest through InstanceNorm2d(affine=False).  Composed from the NHWC BN kernels: batch
    statistics once over all rows, instance statistics per sample, then per-sample scale/shift vectors
    that mix both (so one apply / one dx launch per sample covers all channels)."""

    @staticmethod
    def forward(ctx, x, gamma_bn, beta_bn, running_mean, running_var, training, momentum, eps, group):
        _chk(x, 'x', cl=True)
        b, C, H, W = x.shape
        nb = gamma_bn.numel()
        hw, dev = H * W, x.device
        if not training:
            raise NotImplementedError('IBNorm eval mode is not on the training path')
        sums_all = torch.zeros(2 * C, dtype=torch.float64, device=dev)
        call('pxl_bn_stats', _p(x), b * hw, C, _p(sums_all), _stream())
        sums_i = torch.zeros((b, 2 * C), dtype=torch.float64, device=dev)
        for i in range(b):
            call('pxl_bn_stats', _p(x[i]), hw, C, _p(sums_i[i]), _stream())
        count_all = float(b * hw)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(sums_all, group=group)
            count_all *= dist.get_world_size(group)
        ratio = hw / count_all
        mix = sums_i.clone()
        mix[:, :nb] = sums_all[:nb] * ratio
        mix[:, C:C + nb] = sums_all[C:C + nb] * ratio
        gamma = torch.cat((gamma_bn.detach(), torch.ones(C - nb, device=dev)))
        beta = torch.cat((beta_bn.detach(), torch.zeros(C - nb, device=dev)))
        coeff = torch.empty((b, 4, C), dtype=torch.float32, device=dev)       # mean, invstd, scale, shift per sample
        y = torch.empty_like(x)
        for i in range(b):
            call('pxl_bn_finalize', _p(mix[i]), float(hw), C, _p(gamma), _p(beta), _p(None), _p(None), 0.0, float(eps), 0,
                 _p(coeff[i, 0]), _p(coeff[i, 1]), _p(coeff[i, 2]), _p(coeff[i, 3]), _stream())
            call('pxl_bn_apply', _p(x[i]), _p(coeff[i, 2]), _p(coeff[i, 3]), _p(None), 0, _p(y[i]), hw, C, _stream())
        # running statistics of the BN half (unbiased variance over all rows)
        bn_sums = torch.cat((sums_all[:nb], sums_all[C:C + nb])).contiguous()
        scratch = torch.empty((4, nb), dtype=torch.float32, device=dev)
        call('pxl_bn_finalize', _p(bn_sums), count_all, nb, _p(gamma_bn), _p(beta_bn), _p(running_mean), _p(running_var),
             float(momentum), float(eps), 0, _p(scratch[0]), _p(scratch[1]), _p(scratch[2]), _p(scratch[3]), _stream())
        ctx.save_for_backward(x, coeff, gamma)
        ctx.meta = (b, C, hw, nb, count_all, group)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, coeff, gamma = ctx.saved_tensors
        b, C, hw, nb, count_all, group = ctx.meta
        dy = as_cl(dy)
        dev = dy.device
        dsums = torch.zeros((b, 2 * C), dtype=torch.float64, device=dev)
        for i in range(b):
            call('pxl_bn_bwd_reduce', _p(x[i]), _p(None), _p(dy[i]), _p(coeff[i, 0]), _p(coeff[i, 1]), 0, hw, C,
                 _p(dsums[i]), _p(None), _p(None), _stream())
        tot = dsums.sum(0)
        dgamma = tot[C:C + nb].to(torch.float32)
        dbeta = tot[:nb].to(torch.float32)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(tot, group=group)
        ratio = hw / count_all
        mix = dsums.clone()
        mix[:, :nb] = tot[:nb] * ratio
        mix[:, C:C + nb] = tot[C:C + nb] * ratio
        dx = torch.empty_like(x)
        for i in range(b):
            call('pxl_bn_bwd_dx', _p(x[i]), _p(None), _p(dy[i]), _p(coeff[i, 0]), _p(coeff[i, 1]), _p(gamma), _p(mix[i]),
                 float(hw), 0, _p(dx[i]), _p(None), hw, C, _p(None), _p(None), _p(None), _p(None), _stream())
        return dx, dgamma, dbeta, None, None, None, None, None, None


def ibnorm(x, gamma_bn, beta_bn, running_mean, running_var, training=True, momentum=0.1, eps=1e-5, group=None):
    return _IBNorm.apply(x, gamma_bn, beta_bn, running_mean, running_var, bool(training), float(momentum), float(eps), group)


def gct_dcgt(l_pred, r_pred, l_fm, r_fm, thr):
    """DCGTGenerator.forward (ssl_gct.py:668-689) -> (l_dc_gt, r_dc_gt, both_bad[n,1,H,W])."""
    _chk(l_pred, 'l_pred'); _chk(r_pred, 'r_pred'); _chk(l_fm, 'l_fm'); _chk(r_fm, 'r_fm')
    n, c, h, w = l_pred.shape
    l_dc, r_dc = torch.empty_like(l_pred), torch.empty_like(r_pred)
    both = torch.empty((n, 1, h, w), dtype=torch.float32, device=l_pred.device)
    call('pxl_gct_dcgt', _p(l_pred), _p(r_pred), _p(l_fm), _p(r_fm), float(thr), n, c, h * w, _p(l_dc), _p(r_dc), _p(both),
         _stream())
    return l_dc, r_dc, both


def odd_ksize(v):
    k = int(v)
    return k + 1 if k % 2 == 0 else k


def flawmap_handle(flawmap, im_size, clip_threshold=0.1):
    """FlawmapHandler.forward (ssl_gct.py:641-657): clamp negatives to 0, Gaussian blur
    k = odd(im_size/16), zero the whole map when its max <= 0.1 (min/max taken before), min-max
    normalise.  NOTE: like the reference this also clamps the INPUT tensor's values in place
    (``flawmap.data.mul_(flawmap >= 0)``), which later changes the flaw-detector loss."""
    fm = flawmap.detach()
    fm.clamp_(min=0)                                  # in place on the shared storage, as the reference does
    blurred = gaussian_blur(fm.contiguous(), odd_ksize(im_size / 16))
    return minmax_norm(blurred, 1e-9, clip_threshold)


def fdgt_generate(prob, labels, im_size, mu, nu):
    """FDGTGenerator.forward (ssl_gct.py:714-728) on softmax ``prob`` [n,C,H,W] and float labels [n,1,H,W]."""
    _chk(prob, 'prob'); _chk(labels, 'labels')
    n, c, h, w = prob.shape
    diff = torch.empty((n, 1, h, w), dtype=torch.float32, device=prob.device)
    call('pxl_fdgt_absdiff', _p(prob), _p(labels), float(mu), n, c, h * w, _p(diff), _stream())
    diff = gaussian_blur(diff, odd_ksize(im_size / 8))
    for _ in range(int(nu)):
        diff = gaussian_blur(dilate3x3_reflect(diff), odd_ksize(im_size / 4))
    return minmax_norm(diff, 1e-9, -1.0)


# ------------------------------------------------------------------------------------------------
# CCT / PSPNet decoder pieces
# ------------------------------------------------------------------------------------------------

class _PixelShuffle2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, C, ldo):
        _chk(x, 'x', cl=True)
        n, ldi, h, w = x.shape
        out = torch.empty((n, ldo, 2 * h, 2 * w), dtype=torch.float32, device=x.device, memory_format=CL)
        call('pxl_pixel_shuffle2_nhwc', _p(x), _p(out), n, h, w, C, ldi, ldo, 0, _stream())
        ctx.meta = (n, h, w, C, ldi, ldo)
        return out

    @staticmethod
    def backward(ctx, g):
        n, h, w, C, ldi, ldo = ctx.meta
        g = as_cl(g)
        dx = torch.empty((n, ldi, h, w), dtype=torch.float32, device=g.device, memory_format=CL)
        call('pxl_pixel_shuffle2_nhwc', _p(g), _p(dx), n, h, w, C, ldi, ldo, 1, _stream())
        return dx, None, None


def pixel_shuffle2(x, out_channels, ldo=None):
    """nn.PixelShuffle(2) on a channels_last tensor whose first 4*out_channels lanes are real; the
    result has ``ldo`` lanes (default: out_channels rounded up to 32) with zeros beyond out_channels."""
    if ldo is None:
        ldo = (out_channels + 31) // 32 * 32
    return _PixelShuffle2.apply(as_cl(x), int(out_channels), int(ldo))


class _Perturb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, pixel_mask, chan_scale, elem_noise):
        _chk(x, 'x', cl=True)
        n, c, h, w = x.shape
        out = torch.empty_like(x)
        call('pxl_perturb_nhwc', _p(x), _p(pixel_mask), _p(chan_scale), _p(elem_noise), _p(out), n, h * w, c, _stream())
        ctx.save_for_backward(pixel_mask, chan_scale, elem_noise)
        ctx.meta = (n, c, h, w)
        return out

    @staticmethod
    def backward(ctx, g):
        pixel_mask, chan_scale, elem_noise = ctx.saved_tensors
        n, c, h, w = ctx.meta
        g = as_cl(g)
        dx = torch.empty_like(g)
        call('pxl_perturb_nhwc', _p(g), _p(pixel_mask), _p(chan_scale), _p(elem_noise), _p(dx), n, h * w, c, _stream())
        return dx, None, None, None


def perturb(x, pixel_mask=None, chan_scale=None, elem_noise=None):
    """x * pixel_mask[n,1,H,W] * chan_scale[n,C] * (1 + elem_noise[C,H,W]) on a channels_last feature map
    (CCT perturbations, ssl_cct.py:588, 651, 700-707, 726-727, 743-744).  elem_noise is given in the
    reference's [C,H,W] order and re-laid out to NHWC here."""
    if pixel_mask is not None:
        pixel_mask = pixel_mask.contiguous()
    if chan_scale is not None:
        chan_scale = chan_scale.contiguous()
    if elem_noise is not None:
        elem_noise = elem_noise.permute(1, 2, 0).contiguous()
    return _Perturb.apply(as_cl(x), pixel_mask, chan_scale, elem_noise)


def channel_mean(x):
    """torch.mean(x, dim=1, keepdim=True) of a channels_last tensor -> [n,1,H,W] (no autograd)."""
    _chk(x, 'x', cl=True)
    n, c, h, w = x.shape
    out = torch.empty((n, 1, h, w), dtype=torch.float32, device=x.device)
    call('pxl_channel_mean_nhwc', _p(x), _p(out), n * h * w, c, _stream())
    return out


def argmax_nonzero_mask(logits):
    """(logits.argmax(1) > 0).float() -> [n,1,H,W] for planar logits."""
    _chk(logits, 'logits')
    n, c, h, w = logits.shape
    out = torch.empty((n, 1, h, w), dtype=torch.float32, device=logits.device)
    call('pxl_argmax_nonzero_mask', _p(logits), _p(out), n, c, h * w, _stream())
    return out


class _AdaptiveAvgPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, bin_size):
        _chk(x, 'x', cl=True)
        n, c, h, w = x.shape
        y = torch.empty((n, c, bin_size, bin_size), dtype=torch.float32, device=x.device, memory_format=CL)
        call('pxl_adaptive_avgpool_nhwc', _p(x), _p(y), n, h, w, c, bin_size, 0, _stream())
        ctx.meta = (n, c, h, w, bin_size)
        return y

    @staticmethod
    def backward(ctx, g):
        n, c, h, w, bin_size = ctx.meta
        g = as_cl(g)
        dx = torch.empty((n, c, h, w), dtype=torch.float32, device=g.device, memory_format=CL)
        call('pxl_adaptive_avgpool_nhwc', _p(g), _p(dx), n, h, w, c, bin_size, 1, _stream())
        return dx, None


def adaptive_avg_pool(x, bin_size):
    """nn.AdaptiveAvgPool2d(bin_size) on a channels_last tensor (_pspnet.py:90)."""
    return _AdaptiveAvgPool.apply(as_cl(x), int(bin_size))


class _PyramidConcat(torch.autograd.Function):
    """torch.cat([features] + [F.interpolate(branch, (h, w), 'bilinear', align_corners=False) ...], 1)
    (_pspnet.py:96-101) written straight into one NHWC buffer."""

    @staticmethod
    def forward(ctx, features, *branches):
        _chk(features, 'features', cl=True)
        n, c0, H, W = features.shape
        chans = [c0] + [b.shape[1] for b in branches]
        ld = sum(chans)
        out = torch.empty((n, ld, H, W), dtype=torch.float32, device=features.device, memory_format=CL)
        call('pxl_copy_lanes_nhwc', _p(features), _p(out), n * H * W, c0, ld, 0, 0, _stream())
        off = c0
        for b in branches:
            _chk(b, 'branch', cl=True)
            call('pxl_bilinear_nhwc', _p(b), _p(out), n, b.shape[2], b.shape[3], b.shape[1], H, W, ld, off, 0, 0, _stream())
            off += b.shape[1]
        ctx.meta = (n, H, W, ld, chans, [tuple(b.shape[2:]) for b in branches])
        return out

    @staticmethod
    def backward(ctx, g):
        n, H, W, ld, chans, sizes = ctx.meta
        g = as_cl(g)
        dev = g.device
        df = torch.empty((n, chans[0], H, W), dtype=torch.float32, device=dev, memory_format=CL)
        call('pxl_copy_lanes_nhwc', _p(g), _p(df), n * H * W, chans[0], ld, 0, 1, _stream())
        grads, off = [df], chans[0]
        for c, (h, w) in zip(chans[1:], sizes):
            db = torch.empty((n, c, h, w), dtype=torch.float32, device=dev, memory_format=CL)
            call('pxl_bilinear_nhwc', _p(g), _p(db), n, h, w, c, H, W, ld, off, 0, 1, _stream())
            grads.append(db)
            off += c
        return tuple(grads)


def pyramid_concat(features, branches):
    return _PyramidConcat.apply(as_cl(features), *[as_cl(b) for b in branches])


def confusion_matrix_(cmat, pred, gt, num_classes=None):
    """cmat[gt*C + argmax(pred,1)] += 1 over pixels with 0 <= gt < C, accumulated in place into the int64
    device tensor ``cmat`` [C,C] (task/sseg/func.py:36-48: np.argmax + np.bincount)."""
    _chk(pred, 'pred')
    _chk(gt, 'gt')
    n, c, h, w = pred.shape
    if num_classes is not None and num_classes != c:
        raise ValueError('pred has %d channels, num_classes = %d' % (c, num_classes))
    if gt.numel() != n * h * w:
        raise ValueError('gt must hold one label per pixel')
    if cmat.dtype != torch.int64 or not cmat.is_cuda or cmat.numel() != c * c or not cmat.is_contiguous():
        raise TypeError('cmat must be a contiguous CUDA int64 tensor with C*C entries')
    call('pxl_confusion_matrix', _p(pred), _p(gt), n, c, h * w, ctypes.c_void_p(cmat.data_ptr()), _stream())
    return cmat


_GN_WS = {}


def gaussian_noise_(inp, std, noise=None):
    """GaussianNoiseLayer.forward (pixelssl/nn/module/gaussian_noise.py:18-41) in place on ``inp``
    [n,C,H,W]: noise ~ N(0, uniform(0, std)) drawn by torch's device generator unless given."""
    if std is None:
        return inp
    _chk(inp, 'inp')
    n = inp.shape[0]
    if noise is None:
        import random
        noise = torch.empty_like(inp).normal_(0, std=random.uniform(0, std))
    else:
        _chk(noise, 'noise')
        if noise.shape != inp.shape:
            raise ValueError('noise shape mismatch')
    key = (inp.device.index, n)
    ws = _GN_WS.get(key)
    if ws is None:
        nbytes = _lib.load().pxl_gaussian_noise_workspace_bytes(n)
        ws = _GN_WS[key] = torch.empty(nbytes // 4, dtype=torch.float32, device=inp.device)
    call('pxl_gaussian_noise', _p(inp), _p(noise), n, inp.numel() // n, _p(ws), _stream())
    return inp
