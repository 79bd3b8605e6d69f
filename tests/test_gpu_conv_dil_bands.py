"""The SI-Net's 32-channel 3x3 layers (src/siNet.py:9-10,29-39) on the row-band kernel (csrc/conv_dil.cu), which issues
its MMAs per input band into a ring of eight TMEM accumulator slots: chains longer than the ring, units of one and two
rows, images shorter than the dilation, widths below one 128-pixel tile, the first layer with 6 live input channels,
and one launch per layer.  Each case is held against float64 on the operands the kernel consumed and against the
tap-streaming kernel."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _run(n, hh, ww, dil, terms, seed, live=32, flags=0):
    from dsin_b200 import ops
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, hh, ww, 32)).astype(np.float32)
    x[..., live:] = 0
    w = (rng.standard_normal((3, 3, 32, 32)) / np.sqrt(9 * live)).astype(np.float32)
    bias = (0.3 * rng.standard_normal(32)).astype(np.float32)
    layer = ops.ConvLayer(w, None, bias, dilation=dil, act=ops.ACT_LRELU02)
    layer.flags = flags
    tcl = ops.ConvTC(layer)
    xs = ops.f32_to_split(torch.tensor(x).cuda(), with_lo=terms == 3)
    l0 = ops.launch_count()
    got = ops.conv_tc(xs, tcl, terms=terms)
    launches = ops.launch_count() - l0
    old = ops.conv_tc(xs, tcl, terms=terms, flags=ops.CONV_NO_HALO)
    got = ops.split_to_f32(*got).double()
    old = ops.split_to_f32(*old).double()
    xq = ops.split_to_f32(*xs).double().permute(0, 3, 1, 2)
    w64 = torch.tensor(w, dtype=torch.float64, device="cuda").permute(3, 2, 0, 1)  # [cout][cin][ky][kx]
    ref = F.conv2d(xq, w64, padding=dil, dilation=dil) + torch.tensor(bias, dtype=torch.float64, device="cuda").view(1, -1, 1, 1)
    ref = torch.maximum(0.2 * ref, ref).permute(0, 2, 3, 1)
    return got, old, ref, launches


def _check(got, old, ref, terms):
    tol = (1e-5 if terms == 3 else 4e-3) * max(1.0, float(ref.abs().max()))
    assert float((got - ref).abs().max()) < tol, float((got - ref).abs().max())
    assert float((got - old).abs().max()) < 2 * tol


@pytest.mark.parametrize("terms", [3, 1])
@pytest.mark.parametrize("shape,dil", [
    ((12, 107, 1224), 8),   # 960 units: one segment per chain, chains of 13 and 14 rows (longer than the ring, not x 8)
    ((9, 100, 200), 10),    # 180 units x 5 segments: units of two rows
    ((1, 40, 48), 8),       # units of one row
    ((2, 20, 70), 32),      # H < d: no vertical neighbour inside the image
    ((3, 21, 1224), 1),     # d = 1: bands of 130 pixels, chains of consecutive rows
])
def test_band_kernel_chains_and_units(shape, dil, terms):
    n, hh, ww = shape
    got, old, ref, launches = _run(n, hh, ww, dil, terms, seed=hh + dil)
    assert launches == 1
    _check(got, old, ref, terms)


@pytest.mark.parametrize("terms", [3, 1])
@pytest.mark.parametrize("dil", [1, 2, 4])
@pytest.mark.parametrize("shape", [(2, 40, 48), (1, 37, 100), (1, 9, 20)])
def test_small_dilations_below_one_tile_width(shape, dil, terms):
    n, hh, ww = shape
    got, old, ref, launches = _run(n, hh, ww, dil, terms, seed=3 * hh + dil)
    assert launches == 1
    _check(got, old, ref, terms)


@pytest.mark.parametrize("terms", [3, 1])
@pytest.mark.parametrize("shape", [(2, 40, 48), (1, 320, 1224)])
def test_first_layer_with_six_live_channels(shape, terms):
    """The SI-Net's first layer: 6 live input channels zero-padded to 32.  With CONV_CIN16 the kernel may skip the K-step
    of channels 16..31; the result is the same as without the flag (it only drops products of zeros) and matches
    float64."""
    from dsin_b200 import ops
    n, hh, ww = shape
    got, old, ref, launches = _run(n, hh, ww, 1, terms, seed=hh, live=6, flags=ops.CONV_CIN16)
    assert launches == 1
    _check(got, old, ref, terms)
    full, _, _, _ = _run(n, hh, ww, 1, terms, seed=hh, live=6)
    assert torch.equal(got, full)


def test_one_launch_per_sinet_layer():
    """Every 3x3 layer of the SI-Net (dilations 1, 2, 4, ..., 128, 1) is one kernel launch at full size."""
    from dsin_b200 import ops, siNet as sn
    for li, rate in enumerate(sn.SiNet.RATES):
        _, _, _, launches = _run(1, 320, 1224, rate, 3, seed=li, live=6 if li == 0 else 32,
                                 flags=ops.CONV_CIN16 if li == 0 else 0)
        assert launches == 1, (li, rate, launches)
