"""Thin torch-tensor wrappers over the C ABI (include/dsin_b200.h).

torch is used for device memory and streams only; every arithmetic op below is a kernel of
libdsin_b200.so launched on torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import ACT_LRELU02, ACT_NONE, ACT_RELU, POST_DENORM, POST_DENORM_CLIP, POST_NONE, ConvDesc  # noqa: F401

POST_DENORM_CLIP_D2S = 3

_handles = {}


def handle(device=None):
    if not torch.cuda.is_available():
        raise _lib.DsinLibraryError("CUDA device required: dsin_b200 has no CPU fallback")
    dev = torch.cuda.current_device() if device is None else int(device)
    if dev not in _handles:
        _handles[dev] = _lib.Handle(dev)
    return _handles[dev]


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _chk(t, dtype=torch.float32):
    assert t.is_cuda and t.is_contiguous() and t.dtype == dtype, (t.device, t.is_contiguous(), t.dtype)
    return t


def concat_normalize_split32(xdec_nhwc, ysyn_nhwc, with_lo=True):
    h = handle()
    n, hh, ww, _ = xdec_nhwc.shape
    hi = torch.empty((n, hh, ww, 32), dtype=torch.float16, device=xdec_nhwc.device)
    lo = torch.empty((n, hh, ww, 32), dtype=torch.float16, device=xdec_nhwc.device) if with_lo else None
    h.check(h.lib.dsin_concat_normalize_split32(h.ptr, _p(_chk(xdec_nhwc)), _p(_chk(ysyn_nhwc)), _p(hi), _p(lo), n,
                                                hh, ww, _stream()))
    return hi, lo


def nchw_to_s2d_split32(x, with_lo=True):
    """(n,3,H,W) fp32 image -> normalised space-to-depth(2) split-fp16 (n,H/2,W/2,32) pair."""
    h = handle()
    n, c, hh, ww = x.shape
    assert c == 3 and hh % 2 == 0 and ww % 2 == 0
    hi = torch.empty((n, hh // 2, ww // 2, 32), dtype=torch.float16, device=x.device)
    lo = torch.empty((n, hh // 2, ww // 2, 32), dtype=torch.float16, device=x.device) if with_lo else None
    h.check(h.lib.dsin_nchw_to_s2d_split32(h.ptr, _p(_chk(x)), _p(hi), _p(lo), n, hh, ww, _stream()))
    return hi, lo


class _Profiler(object):
    """Optional per-kernel CUDA-event timing (bench.py's roofline): when enabled every wrapped
    launch is bracketed by events on the launching stream and tagged with its algorithmic FLOPs."""

    def __init__(self):
        self.enabled = False
        self.records = []

    def start(self):
        self.enabled, self.records = True, []

    def stop(self):
        self.enabled = False

    def begin(self):
        if not self.enabled:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def end(self, e0, name, flops=0.0, bytes_=0.0):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self.records.append((name, e0, e1, flops, bytes_))

    def summary(self):
        """name -> dict(ms, launches, flops, bytes); call after a device synchronise."""
        out = {}
        for name, e0, e1, fl, by in self.records:
            d = out.setdefault(name, dict(ms=0.0, launches=0, flops=0.0, bytes=0.0))
            d["ms"] += e0.elapsed_time(e1)
            d["launches"] += 1
            d["flops"] += fl
            d["bytes"] += by
        return out


PROF = _Profiler()


def launch_count():
    return sum(h.launch_count() for h in _handles.values())


def nchw_to_nhwc(x, normalize=False):
    h = handle()
    n, c, hh, ww = x.shape
    y = torch.empty((n, hh, ww, c), dtype=torch.float32, device=x.device)
    h.check(h.lib.dsin_nchw_to_nhwc(h.ptr, _p(_chk(x)), _p(y), n, c, hh, ww, int(normalize), _stream()))
    return y


def nhwc_to_nchw(x):
    h = handle()
    n, hh, ww, c = x.shape
    y = torch.empty((n, c, hh, ww), dtype=torch.float32, device=x.device)
    h.check(h.lib.dsin_nhwc_to_nchw(h.ptr, _p(_chk(x)), _p(y), n, c, hh, ww, _stream()))
    return y


def concat_normalize(xdec_nhwc, ysyn_nhwc):
    h = handle()
    n, hh, ww, _ = xdec_nhwc.shape
    out = torch.empty((n, hh, ww, 6), dtype=torch.float32, device=xdec_nhwc.device)
    h.check(h.lib.dsin_concat_normalize(h.ptr, _p(_chk(xdec_nhwc)), _p(_chk(ysyn_nhwc)), _p(out), n, hh, ww,
                                        _stream()))
    return out


class ConvLayer(object):
    """Device-resident packed parameters of one conv (+ folded BN or bias)."""

    def __init__(self, w_kkio, scale, shift, stride=1, dilation=1, transposed=False, act=ACT_NONE,
                 post=POST_NONE, device="cuda"):
        w = np.ascontiguousarray(w_kkio, dtype=np.float32)
        self.kh, self.kw, self.cin, self.cout = w.shape
        self.w = torch.from_numpy(w).to(device)
        self.scale = None if scale is None else torch.from_numpy(np.ascontiguousarray(scale, np.float32)).to(device)
        self.shift = None if shift is None else torch.from_numpy(np.ascontiguousarray(shift, np.float32)).to(device)
        self.stride, self.dilation, self.transposed, self.act, self.post = stride, dilation, transposed, act, post
        self.dilation_x = 0  # tensor-core path only: tap spacing along W if different from `dilation`
        self.flags = 0       # DSIN_CONV_* flags (tensor-core path only)

    def out_hw(self, hh, ww):
        if self.transposed:
            return 2 * hh, 2 * ww
        return -(-hh // self.stride), -(-ww // self.stride)


def conv2d(x, layer, res1=None, res2=None, scale=None, shift=None, act=None, post=None):
    """y = post(act(conv(x)*scale + shift) + res1 + res2), NHWC fp32."""
    h = handle()
    n, hh, ww, cin = x.shape
    assert cin == layer.cin, (cin, layer.cin)
    oh, ow = layer.out_hw(hh, ww)
    y = torch.empty((n, oh, ow, layer.cout), dtype=torch.float32, device=x.device)
    d = ConvDesc(n, hh, ww, cin, layer.cout, layer.kh, layer.kw, layer.stride, layer.dilation,
                 int(layer.transposed), layer.act if act is None else act, layer.post if post is None else post, 0, 0)
    sc = layer.scale if scale is None else scale
    sh = layer.shift if shift is None else shift
    if res1 is not None:
        assert res1.shape == y.shape
    if res2 is not None:
        assert res2.shape == y.shape
    e0 = PROF.begin()
    h.check(h.lib.dsin_conv2d(h.ptr, C.byref(d), _p(_chk(x)), _p(layer.w), _p(sc), _p(sh), _p(res1), _p(res2),
                              _p(y), _stream()))
    if e0 is not None:
        pix = n * (hh * ww if layer.transposed else oh * ow)  # direct-form dense MACs
        PROF.end(e0, "conv%dx%d_%dto%d%s%s" % (layer.kh, layer.kw, cin, layer.cout,
                                                "_T" if layer.transposed else ("_s%d" % layer.stride),
                                                "_d" if layer.dilation > 1 else ""),
                 2.0 * pix * layer.kh * layer.kw * cin * layer.cout)
    return y


def f32_to_split(x, with_lo=True):
    """fp32 tensor -> (hi, lo) fp16 planes with x ~= hi + lo (22-bit); with_lo=False: (fp16(x), None)."""
    h = handle()
    hi = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    lo = torch.empty(x.shape, dtype=torch.float16, device=x.device) if with_lo else None
    h.check(h.lib.dsin_f32_to_split(h.ptr, _p(_chk(x)), _p(hi), _p(lo), x.numel(), _stream()))
    return hi, lo


def split_to_f32(hi, lo):
    h = handle()
    y = torch.empty(hi.shape, dtype=torch.float32, device=hi.device)
    h.check(h.lib.dsin_split_to_f32(h.ptr, _p(_chk(hi, torch.float16)), _p(lo), _p(y), hi.numel(), _stream()))
    return y


class ConvTC(object):
    """Tensor-core form of a ConvLayer (cin in {32,64,128}, cout <= 128): weights packed
    [tap][npad][cin] as split fp16 with a per-cout power-of-two scale that is folded back into the
    epilogue scale (exact)."""

    def __init__(self, layer):
        assert layer.cin % 32 == 0 and layer.cin <= 128 and layer.cout <= 128, (layer.cin, layer.cout)
        h = handle()
        dev = layer.w.device
        self.layer = layer
        taps = layer.kh * layer.kw
        npad = int(h.lib.dsin_conv_tc_npad(layer.cout))
        self.w_hi = torch.empty((taps, npad, layer.cin), dtype=torch.float16, device=dev)
        self.w_lo = torch.empty((taps, npad, layer.cin), dtype=torch.float16, device=dev)
        wscale = torch.empty((layer.cout,), dtype=torch.float32, device=dev)
        h.check(h.lib.dsin_pack_conv_w_tc(h.ptr, _p(layer.w), taps, layer.cin, layer.cout, _p(self.w_hi),
                                          _p(self.w_lo), _p(wscale), _stream()))
        base = layer.scale if layer.scale is not None else torch.ones_like(wscale)
        self.scale = (base / wscale).contiguous()  # power-of-two division: exact
        self.shift = layer.shift if layer.shift is not None else torch.zeros_like(wscale)
        self.act = layer.act


Conv3x3TC = ConvTC

CONV_PAIR_SHARED = 1
CONV_NO_CTA_PAIR = 2             # cross-check: one-CTA kernel for a 128->128 layer
CONV_NO_WEIGHT_STATIONARY = 4    # cross-check: tap-streaming CTA-pair kernel for a terms = 1 trunk layer
CONV_NO_HALO = 8                 # cross-check: tap-streaming CTA-pair kernel for a terms = 3 trunk layer
CONV_CIN16 = 16                  # 32->32 layer whose input channels 16..31 are zero: skip their K-step


class _PairDesc(object):
    """Geometry of a pixel-pair conv (cin = cout = 64) whose weights are a shared 32x32 slab."""

    def __init__(self, base, rate):
        self.kh, self.kw, self.cin, self.cout = base.kh, base.kw, 64, 64
        self.stride, self.dilation, self.transposed, self.act, self.post = 1, rate, False, base.act, POST_NONE
        self.dilation_x, self.flags = rate // 2, CONV_PAIR_SHARED

    def out_hw(self, hh, ww):
        return hh, ww


class PairSharedTC(object):
    """Even-dilation 32->32 conv applied to pixel pairs: reuses the packed [taps][32][32] weights of the plain
    tensor-core layer; scale/shift are duplicated for the two pixels of a pair."""

    def __init__(self, tcl32, rate):
        assert rate % 2 == 0 and tcl32.layer.cin == 32 and tcl32.layer.cout == 32
        self.layer = _PairDesc(tcl32.layer, rate)
        self.w_hi, self.w_lo = tcl32.w_hi, tcl32.w_lo
        self.scale = torch.cat([tcl32.scale, tcl32.scale]).contiguous()
        self.shift = torch.cat([tcl32.shift, tcl32.shift]).contiguous()
        self.act = tcl32.act



def conv_tc(x, tcl, res1=None, res2=None, terms=3, out_f32=False, post=None, prof=None, flags=0):
    """x: (hi, lo) split-fp16 NHWC pair.  Returns a split pair, or an fp32 NHWC tensor if out_f32.
    terms == 1 (fp16 operands) reads the hi planes only and writes (hi, None): the fp16-operand passes keep
    single-plane fp16 activations, which halves their HBM traffic."""
    h = handle()
    xh, xl = x
    L = tcl.layer
    n, hh, ww, c = xh.shape
    assert c == L.cin
    oh, ow = L.out_hw(hh, ww)
    dev = xh.device
    the_post = L.post if post is None else post
    if out_f32 and the_post == POST_DENORM_CLIP_D2S:  # 12 phase-channels -> (2h, 2w, 3) image
        yf = torch.empty((n, 2 * oh, 2 * ow, 3), dtype=torch.float32, device=dev)
        yh = yl = None
    elif out_f32:
        yf = torch.empty((n, oh, ow, L.cout), dtype=torch.float32, device=dev)
        yh = yl = None
    else:
        yf = None
        yh = torch.empty((n, oh, ow, L.cout), dtype=torch.float16, device=dev)
        yl = torch.empty((n, oh, ow, L.cout), dtype=torch.float16, device=dev) if terms == 3 else None
    r1h, r1l = res1 if res1 is not None else (None, None)
    r2h, r2l = res2 if res2 is not None else (None, None)
    if terms == 3:
        assert xl is not None, "3-term layers need the lo plane of their input"
    d = ConvDesc(n, hh, ww, c, L.cout, L.kh, L.kw, L.stride, L.dilation, int(L.transposed), tcl.act,
                 L.post if post is None else post, int(L.dilation_x), int(getattr(L, "flags", 0)) | int(flags))
    e0 = PROF.begin()
    h.check(h.lib.dsin_conv2d_tc(h.ptr, C.byref(d), terms, _p(_chk(xh, torch.float16)), _p(xl), _p(tcl.w_hi),
                                 _p(tcl.w_lo), _p(tcl.scale), _p(tcl.shift), _p(r1h), _p(r1l), _p(r2h), _p(r2l),
                                 _p(yh), _p(yl), _p(yf), _stream()))
    if e0 is not None and prof is not None:
        PROF.end(e0, prof[0] % terms, prof[1])  # caller-supplied name / algorithmic FLOPs
    elif e0 is not None:
        pix = n * (hh * ww if L.transposed else oh * ow)
        PROF.end(e0, "tc%d_conv%dx%d_%dto%d%s%s" % (terms, L.kh, L.kw, c, L.cout,
                                                     "_T" if L.transposed else ("_s%d" % L.stride),
                                                     "_d" if L.dilation > 1 else ""),
                 2.0 * pix * L.kh * L.kw * c * L.cout)
    return yf if out_f32 else (yh, yl)


def conv3x3_tc(xh, xl, tcl, res1=None, res2=None, terms=3):
    return conv_tc((xh, xl), tcl, res1=res1, res2=res2, terms=terms)


def heatmap_quantize(z33_nhwc, centers, full=False):
    """-> (qbar_nhwc, qbar_nchw, symbols) and, with full=True, also (qhard, z, heatmap), all NCHW."""
    h = handle()
    n, hh, ww, c1 = z33_nhwc.shape
    c = c1 - 1
    dev = z33_nhwc.device
    qbar_nhwc = torch.empty((n, hh, ww, c), dtype=torch.float32, device=dev)
    qbar_nchw = torch.empty((n, c, hh, ww), dtype=torch.float32, device=dev)
    sym = torch.empty((n, c, hh, ww), dtype=torch.int64, device=dev)
    extra = [torch.empty((n, c, hh, ww), dtype=torch.float32, device=dev) for _ in range(3)] if full else [None] * 3
    h.check(h.lib.dsin_heatmap_quantize(h.ptr, _p(_chk(z33_nhwc)), _p(_chk(centers)), centers.numel(), n, hh, ww, c,
                                        _p(qbar_nhwc), _p(qbar_nchw), _p(sym), _p(extra[0]), _p(extra[1]),
                                        _p(extra[2]), _stream()))
    if full:
        return qbar_nhwc, qbar_nchw, sym, extra[0], extra[1], extra[2]
    return qbar_nhwc, qbar_nchw, sym


def probclass_bits(qbar_nchw, symbols, weights, pad_value, k=24, L=6, want_bits=True):
    """weights: list of 4 (w, b) device tensors, mask applied, layout [2][3][3][cin][cout]."""
    h = handle()
    n, c, hh, ww = qbar_nchw.shape
    dev = qbar_nchw.device
    ws = int(h.lib.dsin_probclass_workspace_bytes(n, c, hh, ww, k))
    work = torch.empty(ws, dtype=torch.uint8, device=dev)
    bits = torch.empty((n, c, hh, ww), dtype=torch.float32, device=dev) if want_bits else None
    sums = torch.empty((n,), dtype=torch.float64, device=dev)
    flat = []
    for w, b in weights:
        flat += [_p(_chk(w)), _p(_chk(b))]
    e0 = PROF.begin()
    h.check(h.lib.dsin_probclass_bits(h.ptr, _p(_chk(qbar_nchw)), _p(_chk(symbols, torch.int64)), n, c, hh, ww, k, L,
                                      C.c_float(float(pad_value)), *flat, _p(bits), _p(sums), _p(work), _stream()))
    if e0 is not None:
        vox = lambda a, b_, c_: float(n * (c + a) * (hh + b_) * (ww + c_))  # noqa: E731
        PROF.end(e0, "probclass", 2.0 * 18 * (vox(3, 6, 6) * k + vox(2, 4, 4) * k * k + vox(1, 2, 2) * k * k
                                              + vox(0, 0, 0) * k * L))
    return bits, sums


class ProbclassTC(object):
    """Packed tensor-core weights of the two 24->24 probclass layers (channels zero-padded to 32)."""

    def __init__(self, weights):
        h = handle()
        (w0, b0), (w1, b1), (w2, b2), (w3, b3) = weights
        dev = w0.device
        self.w0, self.b0, self.w3, self.b3 = w0, b0, w3, b3

        def pack(w, b, cout_pad):
            cout = w.shape[-1]
            wp = torch.zeros((18, 32, cout_pad), dtype=torch.float32, device=dev)
            wp[:, :24, :cout] = w.reshape(18, 24, cout)
            bp = torch.zeros((cout_pad,), dtype=torch.float32, device=dev)
            bp[:cout] = b
            npad = int(h.lib.dsin_conv_tc_npad(cout_pad))
            hi = torch.empty((18, npad, 32), dtype=torch.float16, device=dev)
            lo = torch.empty((18, npad, 32), dtype=torch.float16, device=dev)
            ws = torch.empty((cout_pad,), dtype=torch.float32, device=dev)
            h.check(h.lib.dsin_pack_conv_w_tc(h.ptr, _p(wp), 18, 32, cout_pad, _p(hi), _p(lo), _p(ws), _stream()))
            return hi, lo, (1.0 / ws).contiguous(), bp

        self.l1 = pack(w1, b1, 32)
        self.l2 = pack(w2, b2, 32)
        self.l3 = pack(w3, b3, 6)


def probclass_bits_tc(qbar_nchw, symbols, pctc, pad_value, terms=3, want_bits=True):
    h = handle()
    n, c, hh, ww = qbar_nchw.shape
    dev = qbar_nchw.device
    ws = int(h.lib.dsin_probclass_tc_workspace_bytes(n, c, hh, ww))
    work = torch.empty(ws, dtype=torch.uint8, device=dev)
    bits = torch.empty((n, c, hh, ww), dtype=torch.float32, device=dev) if want_bits else None
    sums = torch.empty((n,), dtype=torch.float64, device=dev)
    e0 = PROF.begin()
    h.check(h.lib.dsin_probclass_bits_tc(
        h.ptr, _p(_chk(qbar_nchw)), _p(_chk(symbols, torch.int64)), n, c, hh, ww, C.c_float(float(pad_value)),
        _p(pctc.w0), _p(pctc.b0), _p(pctc.l1[0]), _p(pctc.l1[1]), _p(pctc.l1[2]), _p(pctc.l1[3]),
        _p(pctc.l2[0]), _p(pctc.l2[1]), _p(pctc.l2[2]), _p(pctc.l2[3]),
        _p(pctc.l3[0]), _p(pctc.l3[1]), _p(pctc.l3[2]), _p(pctc.l3[3]), terms,
        _p(bits), _p(sums), _p(work), _stream()))
    if e0 is not None:
        vox = lambda a, b_, c_: float(n * (c + a) * (hh + b_) * (ww + c_))  # noqa: E731
        PROF.end(e0, "probclass_tc%d" % terms, 2.0 * 18 * (vox(3, 6, 6) * 24 + vox(2, 4, 4) * 576 + vox(1, 2, 2) * 576
                                                           + vox(0, 0, 0) * 144))
    return bits, sums


def sif_prepare(xdec_nhwc, ydec_nhwc, ph, pw, lab=False):
    """Pearson: normalised H1/H2/H3 transform; lab=True: CIELAB of the raw pixels (dsin_sif_prepare_lab)."""
    h = handle()
    n, hh, ww, _ = xdec_nhwc.shape
    dev = xdec_nhwc.device
    P = (hh // ph) * (ww // pw)
    q = torch.empty((n, P, ph * pw * 3), dtype=torch.float32, device=dev)
    r = torch.empty((n, hh, ww, 3), dtype=torch.float32, device=dev)
    pstat = torch.empty((n, P, 4), dtype=torch.float32, device=dev)
    ystat = torch.empty((n, hh - ph + 1, ww - pw + 1, 4), dtype=torch.float32, device=dev)
    fn = h.lib.dsin_sif_prepare_lab if lab else h.lib.dsin_sif_prepare
    h.check(fn(h.ptr, _p(_chk(xdec_nhwc)), _p(_chk(ydec_nhwc)), n, hh, ww, ph, pw, _p(q), _p(r), _p(pstat), _p(ystat),
               _stream()))
    return q, r, pstat, ystat


def sif_prepare_lab(xdec_nhwc, ydec_nhwc, ph, pw):
    return sif_prepare(xdec_nhwc, ydec_nhwc, ph, pw, lab=True)


def sif_match(q, r, pstat, ystat, ph, pw, use_mask=True, method=0, l2=False, work=None):
    """Pearson: argmax of the masked correlation; l2=True: argmin of the masked L2 distance (dsin_sif_match_l2), best
    is then the masked distance at the argmin.  work: optional uint8 workspace of sif_workspace_bytes (read it back
    with sif_work_count)."""
    h = handle()
    n, hh, ww, _ = r.shape
    P = q.shape[1]
    dev = r.device
    if work is None:
        work = torch.empty(sif_workspace_bytes(n, hh, ww, ph, pw, method), dtype=torch.uint8, device=dev)
    assert work.dtype == torch.uint8 and work.numel() >= sif_workspace_bytes(n, hh, ww, ph, pw, method)
    row = torch.empty((n, P), dtype=torch.int32, device=dev)
    col = torch.empty((n, P), dtype=torch.int32, device=dev)
    best = torch.empty((n, P), dtype=torch.float32, device=dev)
    fn = h.lib.dsin_sif_match_l2 if l2 else h.lib.dsin_sif_match
    e0 = PROF.begin()
    h.check(fn(h.ptr, _p(_chk(q)), _p(_chk(r)), _p(_chk(pstat)), _p(_chk(ystat)), n, hh, ww, ph, pw, int(use_mask),
               int(method), _p(row), _p(col), _p(best), _p(work), _stream()))
    if e0 is not None:
        PROF.end(e0, "sif_match_l2" if l2 else "sif_match", 2.0 * n * (hh - ph + 1) * (ww - pw + 1) * P * (ph * pw * 3))
    return row, col, best


def sif_match_l2(q, r, pstat, ystat, ph, pw, use_mask=True, method=0, work=None):
    return sif_match(q, r, pstat, ystat, ph, pw, use_mask=use_mask, method=method, l2=True, work=work)


def sif_workspace_bytes(n, hh, ww, ph, pw, method):
    return int(handle().lib.dsin_sif_workspace_bytes(n, hh, ww, ph, pw, method))


def sif_work_count(work, n, hh, ww, ph, pw):
    """Number of (patch, group) work items the last method-1 sif_match on `work` rescored exhaustively."""
    off = int(handle().lib.dsin_sif_work_count_offset(_p(work), n, hh, ww, ph, pw))
    return int(work[off:off + 4].view(torch.int32).item())


def sif_gather(y_nhwc, row, col, ph, pw):
    h = handle()
    n, hh, ww, _ = y_nhwc.shape
    out = torch.empty_like(y_nhwc)
    h.check(h.lib.dsin_sif_gather(h.ptr, _p(_chk(y_nhwc)), _p(_chk(row, torch.int32)), _p(_chk(col, torch.int32)), n,
                                  hh, ww, ph, pw, _p(out), _stream()))
    return out


def validation_terms(x, x_dec, x_with_si, bitcost, heatmap, squared=False):
    """fp32 CUDA tensors x, x_dec, x_with_si (n, ...) (x_with_si may be None), bitcost, heatmap (n, ...) (heatmap may
    be None) -> (n, 4) float64 CUDA tensor of per-image sums [dist(x_dec, x), |x - x_with_si|, bc, bc * heatmap]."""
    h = handle()
    n = x.shape[0]
    img_elems, sym_elems = x.numel() // n, bitcost.numel() // n
    assert x_dec.shape == x.shape and (x_with_si is None or x_with_si.shape == x.shape)
    assert heatmap is None or heatmap.shape == bitcost.shape
    out = torch.empty((n, 4), dtype=torch.float64, device=x.device)
    h.check(h.lib.dsin_validation_terms(h.ptr, _p(_chk(x)), _p(_chk(x_dec)),
                                        None if x_with_si is None else _p(_chk(x_with_si)), _p(_chk(bitcost)),
                                        None if heatmap is None else _p(_chk(heatmap)), n, img_elems, sym_elems,
                                        1 if squared else 0, _p(out), _stream()))
    return out


MSSSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)  # ms_ssim_np_imgcomp.py:91-92


def msssim_levels(img1, img2, groups, batch, height, width, depth):
    """fp32 CUDA tensors viewed as (groups, batch, height, width, depth) -> (groups, 5, 2) float64 CUDA
    tensor of per-level mean SSIM / mean CS."""
    h = handle()
    dev = img1.device
    assert img1.numel() == img2.numel() == groups * batch * height * width * depth
    ws = int(h.lib.dsin_msssim_workspace_bytes(groups, batch, height, width, depth))
    work = torch.empty(ws, dtype=torch.uint8, device=dev)
    out = torch.empty((groups, 5, 2), dtype=torch.float64, device=dev)
    h.check(h.lib.dsin_msssim(h.ptr, _p(_chk(img1)), _p(_chk(img2)), groups, batch, height, width, depth, _p(out),
                              _p(work), _stream()))
    return out


def msssim(img1_nhwc, img2_nhwc, form="standard"):
    """Per-image MS-SSIM of (N,H,W,C) fp32 CUDA tensors -> float64 numpy (N,).
    form="standard": each image as (1,H,W,C); form="reference_call": the reference's literal
    utils.msssim_x_vs_rec view (H,W,C,1) -> batch=H, height=W, width=C, depth=1 (SURVEY F13)."""
    n, hh, ww, c = img1_nhwc.shape
    if form == "standard":
        lv = msssim_levels(img1_nhwc, img2_nhwc, n, 1, hh, ww, c)
    elif form == "reference_call":
        lv = msssim_levels(img1_nhwc, img2_nhwc, n, hh, ww, c, 1)
    else:
        raise ValueError(form)
    lv = lv.cpu().numpy()
    w = np.array(MSSSIM_WEIGHTS)
    return np.prod(lv[:, :4, 1] ** w[:4], axis=1) * (lv[:, 4, 0] ** w[4])


# ---------------------------------------------------------------------------------------------------------------
# PC1 entropy coder (csrc/pc_codec.cu)
# ---------------------------------------------------------------------------------------------------------------
def _pc_codec_ptrs(wlist):
    import ctypes as C
    arr = (C.c_void_p * 8)(*[t.data_ptr() for t in wlist])
    return arr


def pc_stream_capacity(c, hh, ww, nstreams):
    """Bytes that always hold one stream: <= 16 bits per symbol (every frequency is >= 1 of 65536) + flush."""
    slices = (c + nstreams - 1) // nstreams
    return 2 * slices * hh * ww + 16


def pc_encode(symbols, centers, wlist, nstreams=8, wavefront=False):
    """symbols (n,c,h,w) int64 CUDA -> (bytes (n,nstreams,cap) uint8, sizes (n,nstreams) int64, status int32[1]).
    wavefront=True runs the decoder's wavefront kernel in encode mode (same bytes; cross-check)."""
    h = handle()
    n, c, hh, ww = symbols.shape
    dev = symbols.device
    cap = pc_stream_capacity(c, hh, ww, nstreams)
    out = torch.zeros((n, nstreams, cap), dtype=torch.uint8, device=dev)
    sizes = torch.zeros((n, nstreams), dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(int(h.lib.dsin_pc_codec_workspace_bytes(n, c, hh, ww)), dtype=torch.uint8, device=dev)
    ptrs = _pc_codec_ptrs(wlist)
    fn = h.lib.dsin_pc_encode_wavefront if wavefront else h.lib.dsin_pc_encode
    h.check(fn(h.ptr, _p(_chk(symbols, torch.int64)), n, c, hh, ww, _p(_chk(centers)), int(centers.numel()),
                                 ptrs, int(wlist[1].numel()), nstreams, _p(out), cap, _p(sizes), _p(status), _p(ws),
                                 _stream()))
    return out, sizes, status


def pc_decode(stream_bytes, sizes, shape, centers, wlist):
    """stream_bytes (n,nstreams,cap) uint8 CUDA, sizes (n,nstreams) int64 CUDA -> symbols (n,c,h,w) int64."""
    h = handle()
    n, c, hh, ww = shape
    dev = stream_bytes.device
    nstreams, cap = int(stream_bytes.shape[1]), int(stream_bytes.shape[2])
    sym = torch.zeros((n, c, hh, ww), dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(int(h.lib.dsin_pc_codec_workspace_bytes(n, c, hh, ww)), dtype=torch.uint8, device=dev)
    ptrs = _pc_codec_ptrs(wlist)
    h.check(h.lib.dsin_pc_decode(h.ptr, _p(_chk(stream_bytes, torch.uint8)), cap, _p(_chk(sizes, torch.int64)), n, c, hh, ww,
                                 _p(_chk(centers)), int(centers.numel()), ptrs, int(wlist[1].numel()), nstreams, _p(sym),
                                 _p(status), _p(ws), _stream()))
    return sym
