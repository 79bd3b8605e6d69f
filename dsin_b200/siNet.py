"""SI-Net (/root/reference/src/siNet.py:29-41): 9 dilated 3x3 convs (32 ch, LeakyReLU 0.2, bias,
no normalisation) + 1x1 conv to 3 channels, on libdsin_b200 kernels.

``siNet`` is a callable object so that it can own its weights (the reference's TF variables
live in the graph): ``siNet(input[N,6,H,W]) -> [N,3,H,W]``.  ``siNet.fused(x_dec_nhwc,
y_syn_nhwc)`` additionally fuses the normalise+concat in front (src/AE.py:67-68) and the
de-normalisation behind (src/AE.py:69)."""
from __future__ import annotations

import numpy as np
import torch

from . import ops, synth

# Layer forms (all tcgen05).  Every 3x3 layer runs on the row-band kernel (csrc/conv_dil.cu); it beats the halo-tile
# kernel (csrc/conv_h32.cu) at dilation 1, 2 and 4 too.  With BAND off, the layers with a dilation above HALO_MAX_RATE
# run on the tap-streaming kernel (csrc/conv_tc.cu) in the pixel-pair view instead (PAIR: 128-byte TMA rows;
# PAIR_SHARED: even dilations reuse the plain 32x32 slab for both pixels of a pair), the others stay on the band
# kernel.  Module attributes so that tests can compare the forms against each other; the product never changes them.
BAND = True
PAIR = True
PAIR_SHARED = True
HALO_MAX_RATE = 4


class SiNet(object):
    RATES = (1, 2, 4, 8, 16, 32, 64, 128, 1)

    def __init__(self):
        self.layers = None
        self._tc = None
        self.device = "cuda"

    def clone(self):
        """A fresh instance: every AE owns its SI-Net variables (as every TF graph of the reference does), so
        loading weights into one AE never invalidates what another AE's captured CUDA graphs point at."""
        return type(self)()

    def load_weights(self, W):
        S = synth.SIN
        layers = []
        for i, rate in enumerate(self.RATES):
            sc = S + "g_conv%d" % (i + 1)
            layers.append(ops.ConvLayer(W[sc + "/weights"], None, W[sc + "/biases"], dilation=rate,
                                        act=ops.ACT_LRELU02, device=self.device))
        sc = S + "g_conv_last"
        layers.append(ops.ConvLayer(W[sc + "/weights"], None, W[sc + "/biases"], act=ops.ACT_NONE,
                                    device=self.device))
        self.layers = layers
        self._tc = None
        # first layer with its 6 input channels zero-padded to 32 (tensor-core form)
        w1 = np.zeros((3, 3, 32, 32), dtype=np.float32)
        w1[:, :, :6, :] = W[S + "g_conv1/weights"]
        self._first_padded = ops.ConvLayer(w1, None, W[S + "g_conv1/biases"], dilation=1, act=ops.ACT_LRELU02,
                                           device=self.device)
        self._first_padded.flags = ops.CONV_CIN16  # channels 6..31 of its input are zero
        self._tc_first = None
        # the pixel-pair form of the nine 3x3 layers (only used with BAND = False, see _pair_form) is built on demand
        self._w1_padded, self._variables = w1, W
        self._pair = {}
        self._pair_tc = {}

    def _pair_form(self, li):
        """Even dilations in "pixel pair" form: the NHWC tensor (n,H,W,32) is viewed as (n,H,W/2,64); a tap at x offset
        +-d becomes +-d/2 pairs, and the 32x32 weight slab becomes a block-diagonal 64x64 one (pixel parity is preserved
        by an even shift).  Twice the MMA work (on zeros) but half the TMA rows, which is what bounds the tap-streaming
        kernel on these layers."""
        if li not in self._pair:
            sc = synth.SIN + "g_conv%d" % (li + 1)
            w = self._w1_padded if li == 0 else np.asarray(self._variables[sc + "/weights"], np.float32)
            self._pair[li] = self._pair_layer(w, np.asarray(self._variables[sc + "/biases"], np.float32), self.RATES[li])
        return self._pair[li]

    def _pair_layer(self, w, b, rate):
        """3x3 (32->32, dilation `rate`) conv re-expressed on pixel pairs: out parity p at pair j reads input
        pixel 2j + p + dx, i.e. pair j + floor((p+dx)/2) with parity (p+dx) mod 2.  Even rates keep the parity
        (block-diagonal weights, pair taps at +-rate/2); odd rates mix parities (pair taps at +-(rate+1)/2 ...)."""
        offs = sorted({(p_ + (kx - 1) * rate) // 2 for kx in range(3) for p_ in (0, 1)})
        step = offs[1] - offs[0] if len(offs) > 1 else 1
        assert len(offs) == 3 and offs[2] - offs[1] == step and offs[1] == 0, offs  # symmetric 3-tap pattern
        wp = np.zeros((3, 3, 64, 64), dtype=np.float32)
        for kx in range(3):
            for p_ in (0, 1):
                src = p_ + (kx - 1) * rate
                po, pi = src // 2, src % 2
                wp[:, offs.index(po), pi * 32:(pi + 1) * 32, p_ * 32:(p_ + 1) * 32] += w[:, kx]
        layer = ops.ConvLayer(wp, None, np.concatenate([b, b]), dilation=rate, act=ops.ACT_LRELU02,
                              device=self.device)
        layer.dilation_x = step
        return layer

    def _layers_tc(self, cur, n, hh, ww, terms, post):
        """cur: 32-channel split-fp16 NHWC pair (6 live channels) -> fp32 NHWC (n,hh,ww,3)."""
        if hh < 8 or ww < 16:
            raise ValueError("dsin_b200 SI-Net: image smaller than one 8x16 tensor-core tile")
        if self._tc is None:
            self._tc = [ops.ConvTC(layer) for layer in self.layers[1:]]
        if self._tc_first is None:
            self._tc_first = ops.ConvTC(self._first_padded)
        use_pair = PAIR and ww % 2 == 0 and ww // 2 >= 16
        for li, tcl in enumerate([self._tc_first] + self._tc[:-1]):
            # the plain 32-channel layer runs on the row-band kernel (csrc/conv_dil.cu), chosen by dsin_conv2d_tc
            if not BAND and use_pair and self.RATES[li] > HALO_MAX_RATE:
                key = (li, PAIR_SHARED)
                if key not in self._pair_tc:
                    rate = self.RATES[li]
                    if PAIR_SHARED and li >= 1 and rate % 2 == 0:  # parity-preserving: shared 32x32 slab
                        self._pair_tc[key] = ops.PairSharedTC(self._tc[li - 1], rate)
                    else:
                        self._pair_tc[key] = ops.ConvTC(self._pair_form(li))
                v = tuple(None if t is None else t.view(n, hh, ww // 2, 64) for t in cur)
                o = ops.conv_tc(v, self._pair_tc[key], terms=terms,
                                prof=("tc%d_conv3x3_32to32_pair", 2.0 * n * hh * ww * 9 * (6 if li == 0 else 32) * 32))
                cur = tuple(None if t is None else t.view(n, hh, ww, 32) for t in o)
            else:
                cur = ops.conv_tc(cur, tcl, terms=terms)
        return ops.conv_tc(cur, self._tc[-1], terms=terms, out_f32=True, post=post)

    def __call__(self, input, terms=3):  # noqa: A002 - reference argument name
        """siNet(input[N,6,H,W]) -> [N,3,H,W] (src/siNet.py:29-41); the input is already normalised."""
        n, c, hh, ww = input.shape
        if c != 6:
            raise ValueError("siNet expects 6 input channels, got %d" % c)
        net = ops.nchw_to_nhwc(input.contiguous())
        pad = torch.zeros((n, hh, ww, 32), dtype=torch.float32, device=input.device)  # layout only: 6 -> 32 channels
        pad[..., :6] = net
        return ops.nhwc_to_nchw(self._layers_tc(ops.f32_to_split(pad, with_lo=terms == 3), n, hh, ww, terms, ops.POST_NONE))

    def fused(self, x_dec_nhwc, y_syn_nhwc, terms=3):
        n, hh, ww, _ = x_dec_nhwc.shape
        cur = ops.concat_normalize_split32(x_dec_nhwc, y_syn_nhwc, with_lo=terms == 3)
        out_nhwc = self._layers_tc(cur, n, hh, ww, terms, ops.POST_DENORM)
        out = ops.nhwc_to_nchw(out_nhwc)
        out._dsin_nhwc = out_nhwc
        return out


siNet = SiNet()
