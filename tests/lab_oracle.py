"""CPU restatement of the SI-Finder's L2 + LAB matching mode (ae_config.use_L2andLAB = True).  TEST INFRASTRUCTURE
ONLY: imported by tests, never by the product package.

The mode changes three things of src/siFinder.py (:13-17,28-31,102-103,157-195): the images are mapped to CIELAB
without the normalisation, windows are scored by the squared L2 distance instead of Pearson, and the argMIN is taken.
Everything else (encoder, decoder, probability model, crop_and_resize of the original y, SI-Net) is the Pearson
path's, so this module builds on oracle/dsin_oracle.py and restates only what differs.  The reference code this is
pinned to runs in tests/golden/make_lab_golden.py (tests/golden/lab_pieces_golden.npz, tests/test_lab_golden.py).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle import dsin_oracle as O


def _f32c(v, dt):
    """A Python scalar as the float32 constant TF makes of it, in dtype dt."""
    return torch.tensor(float(np.float32(v)), dtype=dt)


def rgb_to_lab(x):
    """rgb_to_lab (src/siFinder.py:157-195) applied to RAW 0..255 values, as the L2 branch does (:13-17).
    Python scalars are float32 constants.  `** 2.4` and `** (1/3)` are pow(x, float32(2.4)) and
    pow(x, float32(1/3)) evaluated in float64 and rounded once to x.dtype.  The 0/1-mask blends are selects (inputs
    are finite and >= 0: same bits).  The two 3x3 matmuls are left to right without FMA (TF pins no order)."""
    dt = x.dtype
    c = lambda v: _f32c(v, dt)  # noqa: E731
    pw_ = lambda t, e: torch.pow(t.to(torch.float64), float(np.float32(e))).to(dt)  # noqa: E731
    lin = torch.where(x <= c(0.04045), x / c(12.92), pw_((x + c(0.055)) / c(1.055), 2.4))
    R, G, B = lin[..., 0], lin[..., 1], lin[..., 2]
    m = [[0.412453, 0.212671, 0.019334], [0.357580, 0.715160, 0.119193], [0.180423, 0.072169, 0.950227]]
    xyz = [(R * c(m[0][k]) + G * c(m[1][k])) + B * c(m[2][k]) for k in range(3)]
    xyz = [xyz[0] * c(1 / 0.950456), xyz[1] * c(1.0), xyz[2] * c(1 / 1.088754)]
    eps = 6 / 29
    fx, fy, fz = (torch.where(t <= c(eps ** 3), t / c(3 * eps ** 2) + c(4 / 29), pw_(t, 1 / 3)) for t in xyz)
    L = ((fx * c(0.0) + fy * c(116.0)) + fz * c(0.0)) + c(-16.0)
    a = ((fx * c(500.0) + fy * c(-500.0)) + fz * c(0.0)) + c(0.0)
    b = ((fx * c(0.0) + fy * c(200.0)) + fz * c(-200.0)) + c(0.0)
    return torch.stack([L, a, b], dim=-1)


def l2_distances(q, r_hwc, mask=None):
    """The masked squared L2 distance of every patch at every position, (P, h, w) in q.dtype (the L2 branch of
    src/siFinder.py:91-103 and the mask multiply, :20).  Sum x^2, sum y^2 and xy are float64 sums of the q.dtype
    values, each rounded once to q.dtype; then out = (sum_x_square - 2 * xy) + sum_y_square and * mask in q.dtype."""
    dt = q.dtype
    P, ph, pw, C = q.shape
    f64 = torch.float64
    q64 = q.to(f64)
    r = r_hwc.to(f64).permute(2, 0, 1).unsqueeze(0)
    sum_x2 = (q64.reshape(P, -1) ** 2).sum(1).to(dt)
    sum_y2 = F.conv2d(r * r, torch.ones(1, C, ph, pw, dtype=f64))[0, 0].to(dt)
    xy = F.conv2d(r, q64.permute(0, 3, 1, 2).contiguous())[0].to(dt)
    out = (sum_x2.view(-1, 1, 1) - 2 * xy) + sum_y2
    if mask is not None:
        out = out * torch.as_tensor(np.asarray(mask)).to(dt)
    return out


def l2_scores(q, r_hwc, mask, chunk=64):
    """l2_distances and tf.argmin over positions (src/siFinder.py:28-29): the first minimal index (-0 == +0; a
    negative value from cancellation competes like any other).  Returns idx (P,) int64 and the masked distance there
    (P,); the (P, h, w) map is built chunk by chunk."""
    P = q.shape[0]
    idx_out = torch.zeros(P, dtype=torch.int64)
    best_out = torch.zeros(P, dtype=q.dtype)
    for s in range(0, P, chunk):
        e = min(P, s + chunk)
        flat = l2_distances(q[s:e], r_hwc, None if mask is None else mask[s:e]).reshape(e - s, -1)
        idx = torch.argmin(flat, dim=1)
        idx_out[s:e] = idx
        best_out[s:e] = flat.gather(1, idx.view(-1, 1)).view(-1)
    return idx_out, best_out


def score_at_l2(q, r_hwc, mask, p, row, col):
    """Masked L2 distance of patch p at one position, in q.dtype (tests adjudicate near-ties with float64)."""
    ph, pw, _C = q.shape[1:]
    win = r_hwc[row:row + ph, col:col + pw, :]
    qp = q[p]
    v = ((qp * qp).sum() - 2 * (qp * win).sum()) + (win * win).sum()
    if mask is not None:
        v = v * float(mask[p, row, col])
    return float(v)


def si_finder(x_patches, y_hwc, mask, ph, pw, y_dec_hwc, force_rowcol=None):
    """src/siFinder.py:7-53, L2 + LAB branch, batch_size == 1 (the analogue of dsin_oracle.si_finder).
    force_rowcol (test helper): (row, col) int arrays, entries >= 0 override the argmin."""
    q = rgb_to_lab(x_patches)
    r = rgb_to_lab(y_dec_hwc)
    idx, best = l2_scores(q, r, mask)
    ncc_w = y_dec_hwc.shape[1] - pw + 1
    row = (idx // ncc_w).to(torch.int32)
    col = (idx % ncc_w).to(torch.int32)
    if force_rowcol is not None:
        fr, fc = (torch.as_tensor(np.asarray(a)).to(torch.int32) for a in force_rowcol)
        row = torch.where(fr >= 0, fr, row)
        col = torch.where(fc >= 0, fc, col)
    yp = O.crop_and_resize_patches(y_hwc.to(torch.float32).numpy(), row.numpy(), col.numpy(), ph, pw)
    return torch.from_numpy(yp).to(x_patches.dtype), best, q, r, row, col


def si_full_img(x_dec, y, y_dec, ph=20, pw=24, use_mask=True, force_rowcol=None):
    """src/siFull_img.py:5-42 with the L2 + LAB SI-Finder: y_syn NCHW plus (row, col, best) per image."""
    N, C, H, W = x_dec.shape
    mask = O.gaussian_masks(H, W, ph, pw) if use_mask else None
    outs, rows, cols, bests = [], [], [], []
    for n in range(N):
        xp = O.extract_patches(x_dec[n].permute(1, 2, 0), ph, pw)
        frc = None if force_rowcol is None else (force_rowcol[0][n], force_rowcol[1][n])
        yp, best, _q, _r, row, col = si_finder(xp, y[n].permute(1, 2, 0), mask, ph, pw, y_dec[n].permute(1, 2, 0), frc)
        outs.append(O.fold_patches(yp, H, W).permute(2, 0, 1))
        rows.append(row)
        cols.append(col)
        bests.append(best)
    return torch.stack(outs), torch.stack(rows), torch.stack(cols), torch.stack(bests)


def _forward(x, y, W, ph, pw, use_mask, force_symbols_x, force_symbols_y, force_rowcol):
    """AE(y), AE(x), bit cost, L2 SI-Finder and SI-Net (src/AE.py:50-69,150-152) -> the pieces both callers need."""
    _ency, y_dec = O.ae_pass(y, W, force_symbols_y)
    encx, x_dec = O.ae_pass(x, W, force_symbols_x)
    bits = O.probclass_bitcost(encx.qbar, encx.symbols, W)
    y_syn, row, col, best = si_full_img(x_dec, y, y_dec, ph, pw, use_mask, force_rowcol)
    x_with_si = O.denormalize(O.si_net(torch.cat([O.normalize(x_dec), O.normalize(y_syn)], dim=1), W))
    return encx, y_dec, x_dec, bits, y_syn, row, col, best, x_with_si


def reconstruct(x_np, y_np, W, dtype=torch.float32, ph=20, pw=24, use_mask=True, force_symbols_x=None,
                force_symbols_y=None, force_rowcol=None):
    """dsin_oracle.reconstruct (AE.siNet_get_reconstructed) with the L2 + LAB SI-Finder."""
    x, y = O._t(x_np, dtype), O._t(y_np, dtype)
    N, _, H, Wd = x.shape
    with torch.no_grad():
        encx, y_dec, x_dec, bits, y_syn, row, col, best, x_with_si = _forward(
            x, y, W, ph, pw, use_mask, force_symbols_x, force_symbols_y, force_rowcol)
    return O.Reconstruction(y_dec, y_syn, x_dec, x_with_si, O.bitcost_to_bpp(bits, N * H * Wd), encx.symbols, row, col,
                            bits.reshape(N, -1).sum(1), best)


def validation_loss(x_np, y_np, W, dtype=torch.float32, ph=20, pw=24, use_mask=True, si_weight=0.7, beta=500.0,
                    H_target=0.04, distortion="mae", K_psnr=100.0, regularization_factor=0.005,
                    regularization_factor_centers=0.1, force_symbols_x=None, force_symbols_y=None, force_rowcol=None):
    """dsin_oracle.validation_loss (AE.siNet_validate, src/AE.py:76-99,120-131) with the L2 + LAB SI-Finder."""
    x, y = O._t(x_np, dtype), O._t(y_np, dtype)
    with torch.no_grad():
        encx, _y_dec, x_dec, bc, _y_syn, _row, _col, _best, x_with_si = _forward(
            x, y, W, ph, pw, use_mask, force_symbols_x, force_symbols_y, force_rowcol)
        d = O.distortion_to_minimize(x, x_dec, distortion, K_psnr)
        reg_enc = O.regularization_loss(W, "autoencoder/encoder", regularization_factor, regularization_factor_centers)
        reg_dec = O.regularization_loss(W, "autoencoder/decoder", regularization_factor, 0.0)
        total, H_real, H_mask, pc_loss = O.get_loss((1.0 - si_weight) * d, bc, encx.heatmap, beta, H_target,
                                                    reg_enc, reg_dec)
        l_si = torch.abs(x - x_with_si).mean()
        loss = total + si_weight * l_si
    return O.ValidationLoss(float(loss), float(d), float(pc_loss), reg_enc + reg_dec, float(l_si), float(H_real),
                            float(H_mask))
