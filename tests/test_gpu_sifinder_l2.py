"""SI-Finder in its L2 + LAB mode (ae_config.use_L2andLAB = True, src/siFinder.py:13-17,28-31,102-103,157-195) against
the oracle: LAB prepare bit for bit, both scorers with and without the prior, edge cases, and the AE entry points.

A (row, col) that differs from the oracle's must be a float64 near-tie: the two positions' masked distances (float64
LAB images) differ by less than the fp32 granularity of the reference's terms, 8 ulp(max(sum x^2, sum y^2)) times the
larger prior of the two."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import dsin_oracle as O

import lab_oracle as L
import oracle_cache
from parity_utils import make_ae

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "lab_pieces_golden.npz"))


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _pair(H, W, seed):
    from dsin_b200 import synth
    x, y = synth.make_pair(seed, H, W, sigma=2.0, disparity=9, noise=3.0)
    return x[None].astype(np.float32), y[None].astype(np.float32)


def _gpu(x, y_dec, y=None, use_mask=True, method=1, with_work=False):
    from dsin_b200 import ops
    y = y_dec if y is None else y
    xt, yt, ydt = (_nhwc(torch.as_tensor(a, dtype=torch.float32).cuda()) for a in (x, y, y_dec))
    n, hh, ww, _ = xt.shape
    q, r, pstat, ystat = ops.sif_prepare_lab(xt, ydt, 20, 24)
    work = torch.empty(ops.sif_workspace_bytes(n, hh, ww, 20, 24, method), dtype=torch.uint8, device="cuda")
    row, col, best = ops.sif_match_l2(q, r, pstat, ystat, 20, 24, use_mask=use_mask, method=method, work=work)
    y_syn = ops.sif_gather(yt, row, col, 20, 24).permute(0, 3, 1, 2).cpu()
    out = (row.cpu(), col.cpu(), best.cpu(), y_syn)
    if with_work:
        return out, (ops.sif_work_count(work, n, hh, ww, 20, 24) if method == 1 else 0)
    return out


def _oracle(x, y_dec, y=None, use_mask=True):
    y = y_dec if y is None else y
    xt, yt, ydt = (torch.as_tensor(a, dtype=torch.float32) for a in (x, y, y_dec))
    y_syn, row, col, best = L.si_full_img(xt, yt, ydt, use_mask=use_mask)
    return row, col, best, y_syn


def _near_ties_only(x, y_dec, got, ref, use_mask=True):
    """Every differing (row, col) is a float64 near-tie (module docstring); returns the number of differences."""
    row, col = got[0].numpy(), got[1].numpy()
    rr, rc = ref[0].numpy(), ref[1].numpy()
    mism = (row != rr) | (col != rc)
    N, _, H, W = x.shape
    mask = O.gaussian_masks(H, W, 20, 24) if use_mask else None
    for n, p in zip(*np.nonzero(mism)):
        q64 = O.extract_patches(L.rgb_to_lab(torch.as_tensor(x[n], dtype=torch.float64).permute(1, 2, 0)), 20, 24)
        r64 = L.rgb_to_lab(torch.as_tensor(y_dec[n], dtype=torch.float64).permute(1, 2, 0))
        sx2 = float((q64[p] ** 2).sum())
        terms, ms = [sx2], []
        for i, j in ((row[n, p], col[n, p]), (rr[n, p], rc[n, p])):
            terms.append(float((r64[i:i + 20, j:j + 24] ** 2).sum()))
            ms.append(1.0 if mask is None else float(mask[p, i, j]))
        gap = 8 * float(np.spacing(np.float32(max(terms)))) * max(ms)
        a = L.score_at_l2(q64, r64, mask, p, int(row[n, p]), int(col[n, p]))
        b = L.score_at_l2(q64, r64, mask, p, int(rr[n, p]), int(rc[n, p]))
        assert abs(a - b) <= gap, (n, p, a, b, gap)
    return int(mism.sum())


def _agree(x, y_dec, got, ref, use_mask, what):
    """(row, col) equal to the oracle's up to float64 near-ties; y_syn bit-exact on every patch whose (row, col) agree;
    the masked distance at the argmin within 4 ulp of the oracle's there."""
    n = _near_ties_only(x, y_dec, got, ref, use_mask)
    print("%s: %d / %d (row, col) differ from the oracle (float64 near-ties)" % (what, n, ref[0].numel()))
    same = (got[0] == ref[0]) & (got[1] == ref[1])                     # (N, P)
    N, _, H, W = x.shape
    pix = same.reshape(N, H // 20, 1, W // 24, 1).expand(N, H // 20, 20, W // 24, 24).reshape(N, 1, H, W)
    pix = pix.expand(N, 3, H, W)
    assert torch.equal(got[3][pix], ref[3][pix]), what
    g, r = got[2][same].double().numpy(), ref[2][same].double().numpy()
    assert np.all(np.abs(g - r) <= 4 * np.spacing(np.abs(r).astype(np.float32)).astype(np.float64) + 1e-30), what
    return n


# ---------------------------------------------------------------------------------------------------------- prepare
def test_prepare_lab_is_bit_equal_to_the_oracle_and_near_the_reference():
    from dsin_b200 import ops
    x, y = _pair(80, 144, 1)
    x[0, :, :20, :48] = 0.0  # black: both linear branches
    y[0, :, 40:, 100:] = 0.0
    xt, yt = _nhwc(torch.tensor(x).cuda()), _nhwc(torch.tensor(y).cuda())
    q, r, pstat, ystat = ops.sif_prepare_lab(xt, yt, 20, 24)
    q_ref = O.extract_patches(L.rgb_to_lab(torch.tensor(x[0]).permute(1, 2, 0)), 20, 24)
    r_ref = L.rgb_to_lab(torch.tensor(y[0]).permute(1, 2, 0))
    assert torch.equal(q.cpu()[0], q_ref.reshape(q_ref.shape[0], -1))
    assert torch.equal(r.cpu()[0], r_ref)
    # pstat / ystat: sums of squares as fp64 sums rounded once (what the L2 score reads)
    assert torch.equal(pstat.cpu()[0, :, 1], (q_ref.double().reshape(q_ref.shape[0], -1) ** 2).sum(1).float())
    # against the reference's own rgb_to_lab (float32 pow, unpinned matmul order): 4 ulp of the largest term
    gx = torch.tensor(GOLD["l2_x"])[None].cuda()
    gy = torch.tensor(GOLD["l2_y"])[None].cuda()
    q, r, _ps, _ys = ops.sif_prepare_lab(gx.contiguous(), gy.contiguous(), 20, 24)
    for got, want in ((q.cpu().numpy().reshape(-1, 3), GOLD["l2_q"].reshape(-1, 3)),
                      (r.cpu().numpy().reshape(-1, 3), GOLD["l2_r"].reshape(-1, 3))):
        want = want.astype(np.float64)
        fy = (want[:, 0] + 16.0) / 116.0
        fx, fz = fy + want[:, 1] / 500.0, fy - want[:, 2] / 200.0
        terms = [116.0 * fy, 500.0 * np.maximum(fx, fy), 200.0 * np.maximum(fy, fz)]
        for c in range(3):
            ulp = np.spacing(np.abs(terms[c]).astype(np.float32)).astype(np.float64)
            assert np.all(np.abs(got[:, c] - want[:, c]) <= 4 * ulp), c


# ---------------------------------------------------------------------------------------------------------- match
@pytest.mark.parametrize("geom", [(80, 144), (120, 96)])
@pytest.mark.parametrize("use_mask", [False, True])
@pytest.mark.parametrize("method", [0, 1])
def test_match_equals_the_oracle(geom, use_mask, method):
    H, W = geom
    x, y = _pair(H, W, 11 + H)
    got = _gpu(x, y, use_mask=use_mask, method=method)
    ref = _oracle(x, y, use_mask=use_mask)
    _agree(x, y, got, ref, use_mask, "%dx%d mask=%s method=%d" % (H, W, use_mask, method))


def test_the_prior_pulls_matches_to_the_corners():
    """The prior multiplies a distance (src/siFinder.py:20): without it patch 1 finds its disparity-9 match, with it
    most patches go to the far rows / columns -- the reference's behaviour, reproduced, not corrected."""
    x, y = _pair(80, 144, 0)
    free = _gpu(x, y, use_mask=False)
    prior = _gpu(x, y, use_mask=True)
    assert (int(free[0][0, 1]), int(free[1][0, 1])) == (0, 33)
    far = ((prior[0][0, :12] == 60) & ((prior[1][0, :12] <= 2) | (prior[1][0, :12] >= 119))).sum()
    assert int(far) >= 9, (prior[0][0, :12], prior[1][0, :12])


def test_full_size_tcgen05_against_simt_and_the_oracle_on_decoded_images():
    """320x1224 decoded images (the oracle's own decoder outputs): tcgen05 vs the SIMT scorer, and vs the oracle."""
    Wt, d = oracle_cache.get("full1")
    x_dec, y_dec, y = d["ref_x_dec"][:1], d["ref_y_dec"][:1], d["y"][:1].astype(np.float32)
    tc, work = _gpu(x_dec, y_dec, y=y, use_mask=True, method=1, with_work=True)
    simt = _gpu(x_dec, y_dec, y=y, use_mask=True, method=0)
    ref = _oracle(x_dec, y_dec, y=y, use_mask=True)
    print("full size: %d exhaustive work items" % work)
    n1 = _near_ties_only(x_dec, y_dec, tc, (simt[0], simt[1]), True)
    n2 = _agree(x_dec, y_dec, tc, ref, True, "320x1224 decoded, tcgen05")
    print("tcgen05 vs SIMT: %d differ; vs oracle: %d" % (n1, n2))


# ---------------------------------------------------------------------------------------------------------- edges
@pytest.mark.parametrize("use_mask", [False, True])
def test_constant_side_image_ties_every_window(use_mask):
    """y_dec constant: every window has the same distance, bit for bit.  Without the prior tf.argmin takes index 0;
    with it the smallest prior wins, as in the oracle."""
    x, _ = _pair(80, 144, 3)
    y_dec = np.full_like(x, 117.0)
    got = _gpu(x, y_dec, use_mask=use_mask)
    ref = _oracle(x, y_dec, use_mask=use_mask)
    if not use_mask:
        assert int(ref[0].abs().sum()) == 0 and int(ref[1].abs().sum()) == 0
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert torch.equal(got[3], ref[3])


@pytest.mark.parametrize("use_mask", [False, True])
def test_black_regions(use_mask):
    """Black (0) and near-black pixels take the linear branches of both piecewise functions of rgb_to_lab."""
    x, y = _pair(80, 144, 5)
    x[:, :, 20:60, 24:72] = 0.0
    y[:, :, 20:60, 33:81] = 0.0
    y[:, :, :20, :] = np.minimum(y[:, :, :20, :], 1.0)
    got = _gpu(x, y, use_mask=use_mask)
    ref = _oracle(x, y, use_mask=use_mask)
    _agree(x, y, got, ref, use_mask, "black regions mask=%s" % use_mask)


@pytest.mark.parametrize("use_mask", [False, True])
def test_identical_images(use_mask):
    """y = x on texture: without the prior every patch matches itself (distance 0, or a cancellation residue)."""
    x, _ = _pair(80, 144, 9)
    got = _gpu(x, x.copy(), use_mask=use_mask)
    ref = _oracle(x, x.copy(), use_mask=use_mask)
    _agree(x, x, got, ref, use_mask, "y = x mask=%s" % use_mask)
    if not use_mask:
        P = ref[0].shape[1]
        top = torch.tensor([(p // 6) * 20 for p in range(P)], dtype=torch.int32)
        left = torch.tensor([(p % 6) * 24 for p in range(P)], dtype=torch.int32)
        assert torch.equal(got[0][0], top) and torch.equal(got[1][0], left)


@pytest.mark.parametrize("use_mask", [False, True])
def test_periodic_texture_needs_the_exhaustive_pass(use_mask):
    """320x1224, 8-periodic texture (as test_gpu_sifinder_edge): exact ties between periods fill the 4 candidates of a
    group, so groups go on the exhaustive work list; the result still equals the oracle."""
    H, W = 320, 1224
    rng = np.random.default_rng(0)
    xx = np.mgrid[0:H, 0:W][1]
    col_code = rng.uniform(0, 255, size=(3, H, 8))
    img = np.floor(col_code[:, :, xx[0] % 8][None]).astype(np.float32)
    got, work = _gpu(img, img.copy(), use_mask=use_mask, with_work=True)
    ref = _oracle(img, img.copy(), use_mask=use_mask)
    print("periodic mask=%s: %d exhaustive work items" % (use_mask, work))
    assert work > 0
    _agree(img, img, got, ref, use_mask, "periodic 320x1224 mask=%s" % use_mask)


# ---------------------------------------------------------------------------------------------------------- AE level
def _l2_ae(H=80, W=144):
    Wt, d = oracle_cache.get("small")
    ae = make_ae(H, W, Wt)
    ae.ae_config.use_L2andLAB = True
    return ae, Wt, d


def test_ae_eager_equals_graph_replay_and_the_oracle():
    ae, Wt, d = _l2_ae()
    x, y = d["x"], d["y"]
    ae.use_cuda_graph = True
    g = [np.array(a) for a in ae.siNet_get_reconstructed(x, y)]
    g_rc = (ae.last["row"].cpu().clone(), ae.last["col"].cpu().clone())
    ae.use_cuda_graph = False
    e = [np.array(a) for a in ae.siNet_get_reconstructed(x, y)]
    for a, b in zip(g, e):
        assert np.array_equal(a, b)
    assert torch.equal(g_rc[0], ae.last["row"].cpu()) and torch.equal(g_rc[1], ae.last["col"].cpu())
    # against the oracle fed the GPU's own symbols (the quantiser's float64 near-ties are the Pearson tests' business)
    sym_x, sym_y = ae.last["symbols"].cpu(), ae.last["symbols_y"].cpu()
    ref = L.reconstruct(x.astype(np.float32), y.astype(np.float32), Wt, force_symbols_x=sym_x,
                        force_symbols_y=sym_y)
    row, col = g_rc[0].numpy(), g_rc[1].numpy()
    mism = (row != ref.row.numpy()) | (col != ref.col.numpy())
    print("AE L2: %d / %d (row, col) differ from the oracle" % (int(mism.sum()), mism.size))
    assert int(mism.sum()) <= max(2, mism.size // 100)
    fr, fc = np.where(mism, row, -1), np.where(mism, col, -1)
    if mism.any():
        ref = L.reconstruct(x.astype(np.float32), y.astype(np.float32), Wt, force_symbols_x=sym_x,
                            force_symbols_y=sym_y, force_rowcol=(fr, fc))
    worst = float(np.abs(g[3] - ref.x_with_si.numpy()).max())
    print("AE L2: max |d x_with_si| %.3f grey levels" % worst)
    assert worst < 2.0


def test_ae_compress_decompress_and_validate():
    ae, Wt, d = _l2_ae()
    x, y = d["x"], d["y"]
    ae.siNet_get_reconstructed(x, y)
    row, col = ae.last["row"].cpu().clone(), ae.last["col"].cpu().clone()
    streams = ae.compress(x)
    ae.decompress(streams, y)
    assert torch.equal(ae.last["row"].cpu(), row) and torch.equal(ae.last["col"].cpu(), col)
    loss = ae.siNet_validate(x, y)
    c = ae.ae_config
    sym_x, sym_y = ae.last["symbols"].cpu(), ae.last["symbols_y"].cpu()
    ref = L.validation_loss(x.astype(np.float32), y.astype(np.float32), Wt, si_weight=c.si_weight, beta=c.beta,
                            H_target=c.H_target, distortion=c.distortion_to_minimize, K_psnr=c.K_psnr,
                            regularization_factor=c.regularization_factor,
                            regularization_factor_centers=c.regularization_factor_centers,
                            force_symbols_x=sym_x, force_symbols_y=sym_y)
    print("AE L2: loss_test gpu %.7f oracle %.7f" % (loss, ref.loss))
    assert abs(loss - ref.loss) <= 2e-6 * abs(ref.loss)


def test_flipping_the_flag_on_one_ae_gives_each_modes_own_result():
    Wt, d = oracle_cache.get("small")
    x, y = d["x"], d["y"]
    results = {}
    for l2 in (False, True):
        fresh = make_ae(80, 144, Wt)
        fresh.ae_config.use_L2andLAB = l2
        fresh.siNet_get_reconstructed(x, y)
        results[l2] = (fresh.last["row"].cpu().clone(), fresh.last["col"].cpu().clone())
    assert not (torch.equal(results[False][0], results[True][0]) and torch.equal(results[False][1], results[True][1]))
    ae = make_ae(80, 144, Wt)
    for l2 in (True, False, True, False):
        ae.ae_config.use_L2andLAB = l2
        ae.siNet_get_reconstructed(x, y)
        assert torch.equal(ae.last["row"].cpu(), results[l2][0]) and torch.equal(ae.last["col"].cpu(), results[l2][1])
    assert len(ae._graphs) == 2


def test_main_runs_with_the_flag_set(tmp_path):
    src = os.path.join(ROOT, "dsin_b200", "run_configs", "ae_run_configs")
    text = open(src).read()
    assert "use_L2andLAB = False" in text
    cfg = tmp_path / "ae_run_configs"
    cfg.write_text(text.replace("use_L2andLAB = False", "use_L2andLAB = True"))
    cmd = [sys.executable, "-m", "dsin_b200.main", "-ae_config", str(cfg), "-pc_config",
           os.path.join(ROOT, "dsin_b200", "run_configs", "pc_run_configs"), "--synthetic", "2", "--random_init",
           "--no_save_test_img"]
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert out.stdout.count("bpp = ") == 2, out.stdout[-1500:]
