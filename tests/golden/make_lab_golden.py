"""Generates tests/golden/lab_pieces_golden.npz: the SI-Finder's L2 + LAB matching mode (use_L2andLAB = True) as the
reference's own code computes it.

Run from the repository root with a checkout of the reference (ayziksha/DSIN):
    python tests/golden/make_lab_golden.py <path of the DSIN checkout>

The reference's rgb_to_lab, check_image and the LAB branch of rgb_transform (src/siFinder.py:138-210) run on pixel
values that hit both branches of both piecewise functions, and the L2 branch of L2_or_pearson_corr (:76-135) on small
LAB images.  They are extracted with ``ast`` and executed on the numpy stand-in for TensorFlow of make_golden.py,
extended by the ops these functions use: pow, comparisons and matmul in float32 as TF does, Python scalars and lists as
float32 constants, and tf.nn.conv2d as a float64 VALID correlation rounded to float32 (this pins the reference's
algebra and its order, not the convolution).  Nothing from the reference is copied into the repo; only its numeric
outputs are stored.
"""
import ast
import os
import sys
import types

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import OUT, _T, _make_tf, _raw  # noqa: E402

REF = None  # src/ of the DSIN checkout named on the command line


def _make_tf_lab():
    """The stand-in plus the ops rgb_to_lab / check_image / L2_or_pearson_corr use.  Python scalars and lists become
    float32 constants, as in TF."""
    import contextlib
    from numpy.lib.stride_tricks import sliding_window_view
    f32 = np.float32
    tf = _make_tf()

    def conv2d(y, w, strides=None, padding=None):
        assert padding == "VALID" and list(strides) == [1, 1, 1, 1]
        y, w = np.asarray(_raw(y), np.float64), np.asarray(_raw(w), np.float64)  # (N,H,W,C), (kh,kw,C,O)
        win = sliding_window_view(y, w.shape[:2], axis=(1, 2))                    # (N,h,w,C,kh,kw)
        return _T(np.einsum("nijcab,abco->nijo", win, w).astype(f32))

    def constant(v, dtype=None, shape=None, name=None):
        a = np.asarray(v, dtype=dtype.np_dtype if dtype else f32)
        return _T(np.full(shape, a, a.dtype) if shape is not None else a)

    tf.nn.conv2d = conv2d
    tf.constant = constant
    tf.cast = lambda v, dtype: _T(np.asarray(_raw(v)).astype(dtype.np_dtype))
    tf.matmul = lambda a, b: _T(np.matmul(_raw(a), _raw(b)))
    tf.multiply = lambda a, b: _T(np.multiply(_raw(a), np.asarray(_raw(b), f32)))
    tf.transpose = lambda v, perm: _T(np.transpose(_raw(v), perm))
    tf.assert_equal = lambda a, b, message=None: None
    tf.control_dependencies = lambda deps: contextlib.nullcontext()
    tf.identity = lambda v: _T(_raw(v))
    return tf


def make_lab_pieces():
    """LAB transform and L2 score of the use_L2andLAB = True matching mode, from the reference's own code."""
    _T.__pow__ = lambda self, e: _T(np.power(self.a, e))  # float32 ** python float -> float32 (NEP 50), as TF
    _T.__le__ = lambda self, o: _T(self.a <= np.float32(_raw(o)))
    _T.__gt__ = lambda self, o: _T(self.a > np.float32(_raw(o)))
    _T.set_shape = lambda self, shape: None
    tree = ast.parse(open(os.path.join(REF, "siFinder.py")).read())
    names = {"rgb_transform", "rgb_to_lab", "check_image", "L2_or_pearson_corr"}
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
    ns = {"np": np, "tf": _make_tf_lab()}
    exec(compile(ast.Module(body=body, type_ignores=[]), "siFinder.py", "exec"), ns)
    cfg = types.SimpleNamespace(use_L2andLAB=True)
    rng = np.random.default_rng(41)
    f32 = np.float32
    special = np.array([0, 0.01, f32(0.04045), 0.0405, 1, 254.5, 255], np.float32)
    grid = np.stack(np.meshgrid(special, special, special, indexing="ij"), -1).reshape(-1, 3)  # every combination
    rand = rng.uniform(0, 255, size=(512, 3)).astype(np.float32)
    px = np.concatenate([grid, rand, np.floor(rand[:64])]).astype(np.float32)
    out = {"lab_in": px, "lab_out": ns["rgb_transform"](_T(px[None, None]), cfg).a[0, 0]}
    # L2 scores: a 40x48 x image tiled into 20x24 patches against a 40x48 y_dec (textured + a black corner)
    H, W, ph, pw = 40, 48, 20, 24
    yy, xx = np.mgrid[0:H, 0:W]
    base = 128 + 90 * np.sin(2 * np.pi * xx / 13.0) * np.cos(2 * np.pi * yy / 11.0)
    y_img = np.clip(np.stack([base, 0.6 * base + 50, 255 - base], -1) + rng.normal(0, 6, (H, W, 3)), 0, 255)
    y_img[:8, :10] = 0.0
    x_img = np.clip(np.roll(y_img, 5, axis=1) + rng.normal(0, 4, (H, W, 3)), 0, 255)
    x_img, y_img = x_img.astype(np.float32), y_img.astype(np.float32)
    xp = x_img.reshape(H // ph, ph, W // pw, pw, 3).transpose(0, 2, 1, 3, 4).reshape(-1, ph, pw, 3)
    q = ns["rgb_transform"](_T(xp), cfg)
    r = ns["rgb_transform"](_T(y_img[None]), cfg)
    out.update(l2_x=x_img, l2_y=y_img, l2_q=q.a, l2_r=r.a[0], l2_out=ns["L2_or_pearson_corr"](q, r, cfg).a[0])
    np.savez_compressed(os.path.join(OUT, "lab_pieces_golden.npz"), **out)


if __name__ == "__main__":
    REF = os.path.join(sys.argv[1], "src")
    make_lab_pieces()
    print("lab_pieces_golden.npz", os.path.getsize(os.path.join(OUT, "lab_pieces_golden.npz")))
