"""SI-Finder on libdsin_b200 (/root/reference/src/siFinder.py:7-53).

``siFinder(x_patches, y_images, mask, batch_size, ph, pw, H, W, ae_config, y_dec)`` keeps the
reference signature (channel-last tensors).  ``match_images`` is the whole-image entry used
by SI_full_img: it never tiles x into patches on the host and never materialises the
correlation map (``ncc`` is returned as None).

Both matching modes of the reference are built, selected by ``ae_config.use_L2andLAB`` as there:

* False (the shipped config): the images are normalised and mapped to H1/H2/H3, windows are scored by
  Pearson correlation times the Gaussian prior, and the argmax is taken.
* True: the RAW 0..255 pixels are mapped to CIELAB (rgb_to_lab assumes sRGB in [0, 1], so the values come out
  far outside the usual LAB ranges: white has L ~ 9342), windows are scored by the squared L2 distance
  ``(sum_x_square - 2 * xy) + sum_y_square`` times the prior, and the argMIN is taken (first index on ties).
  ``q`` / ``r`` are then the LAB images, ``extremum`` the argmin index and ``best`` the masked distance there.
  Quirk kept from the reference: the prior, a factor in (0, 1] that is largest at the patch's own position,
  MULTIPLIES a distance here, so it makes far-away windows cheaper and pulls the matches toward the image
  corners rather than toward the patch (use_gauss_mask = False avoids it).
"""
from __future__ import annotations

import torch

from . import ops

METHOD = 1  # 0: SIMT scorer (cross-check); 1: tcgen05 coarse scorer + exact rescoring


class GaussianPrior(object):
    """Stand-in for the (1,h,w,P) constant of AE.create_gaussian_masks (src/AE.py:193-220):
    the kernels evaluate the prior analytically, so only its geometry is kept."""

    def __init__(self, H, W, ph, pw):
        self.H, self.W, self.ph, self.pw = H, W, ph, pw


def uses_l2(ae_config):
    """The matching mode ae_config selects: True for L2 + LAB (use_L2andLAB), False for Pearson."""
    return bool(ae_config is not None and getattr(ae_config, "use_L2andLAB", False))


def match_images(x_dec_nhwc, y_nhwc, y_dec_nhwc, ph, pw, use_mask, ae_config=None):
    l2 = uses_l2(ae_config)
    q, r, pstat, ystat = ops.sif_prepare(x_dec_nhwc, y_dec_nhwc, ph, pw, lab=l2)
    row, col, best = ops.sif_match(q, r, pstat, ystat, ph, pw, use_mask=use_mask, method=METHOD, l2=l2)
    y_syn = ops.sif_gather(y_nhwc, row, col, ph, pw)
    return y_syn, q, r, row, col, best


def siFinder(x_patches_orig, y_images_orig, mask, batch_size, patch_size_h, patch_size_w, H, W, ae_config, y_dec):
    if batch_size != 1:
        raise NotImplementedError("reference SI path is batch 1 per call (src/AE.py:26); use match_images")
    ph, pw = patch_size_h, patch_size_w
    # fold the (P,ph,pw,3) patches back to the (1,H,W,3) image they tile (layout only)
    x_img = x_patches_orig.reshape(H // ph, W // pw, ph, pw, 3).permute(0, 2, 1, 3, 4).reshape(1, H, W, 3).contiguous()
    use_mask = isinstance(mask, GaussianPrior)
    y_syn, q, r, row, col, _best = match_images(x_img, y_images_orig.contiguous(), y_dec.contiguous(), ph, pw,
                                                use_mask, ae_config)
    y_patches = y_syn.reshape(H // ph, ph, W // pw, pw, 3).permute(0, 2, 1, 3, 4).reshape(-1, ph, pw, 3)
    ncc_w = W - pw + 1
    extremum = row * ncc_w + col
    return y_patches, None, extremum, q.reshape(-1, ph, pw, 3), r, row, col
