"""Generates tests/golden/*.npz from the parts of the reference that run in this container.

Run from the repository root with a checkout of the reference (ayziksha/DSIN):
    python tests/golden/make_golden.py <path of the DSIN checkout>
  * mask_golden.npz   - AE.create_gaussian_masks (src/AE.py:193-220), extracted with ``ast``
                        and executed with a stub ``self`` (pure numpy).
  * msssim_golden.npz - ms_ssim_np_imgcomp.MultiScaleSSIM / utils.msssim_x_vs_rec call forms
                        (src/ms_ssim_np_imgcomp.py, src/utils.py:94-99) with ``tensorflow``
                        stubbed in sys.modules (the module never uses it).
  * model_pieces_golden.npz - the numpy-only pieces of the model code, extracted with ``ast`` and run with a stub
                        ``tf.name_scope``: the causal conv masks (src/probclass_imgcomp.py:150-176), the symbol
                        volume padding and its inverse (:268-292, :341-353), the block iteration order of the coder
                        helpers (:371-393), AE.normalize / denormalize / get_mean_var (src/AE.py:222-250), and the
                        host helpers readfiles (src/DataProvider.py:96-100), l1_x_vs_rec and save_test_imgs_fn
                        (src/utils.py:82-111).
  * run_configs_golden.json - what src/run_configs/{ae,pc}_run_configs parse to (repr of every value).
  * tf_pieces_golden.npz - reference functions whose bodies are elementwise / shape TensorFlow ops only, extracted with
                        ``ast`` and executed under a small numpy stand-in for those ops (``_make_tf`` / ``_T`` below: tile,
                        expand_dims, split, concat, sigmoid, softmax, argmax, one_hot, reduce_sum, ... each following the
                        op's documented semantics in float32): reduce_mean_and_std_normalize_images and rgb_transform
                        (src/siFinder.py:56-73,138-154), _get_heatmap3D and _mask_with_heatmap
                        (src/autoencoder_imgcomp.py:173-201), _quantize1d and phi_times_centers
                        (src/quantizer_imgcomp.py:43-100), bitcost_to_bpp (src/bits_imgcomp.py:4-20).  This pins which
                        channels / constants / formulas the reference's own code applies; the convolution-type ops
                        (Conv2D, Conv3D, CropAndResize, ExtractImagePatches) have no stand-in and stay unpinned.
Nothing from the reference is copied into the repo; only its numeric outputs are stored.
"""
import ast
import json
import os
import sys
import types

import numpy as np

REF = None  # src/ of the DSIN checkout named on the command line
OUT = os.path.dirname(os.path.abspath(__file__))


def reference_mask_fn():
    src = open(os.path.join(REF, "AE.py")).read()
    tree = ast.parse(src)
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "create_gaussian_masks":
            mod = ast.Module(body=[node], type_ignores=[])
            ns = {"np": np}
            exec(compile(mod, "AE.create_gaussian_masks", "exec"), ns)
            return ns["create_gaussian_masks"]
    raise RuntimeError("create_gaussian_masks not found")


def make_masks():
    fn = reference_mask_fn()
    out = {}
    for (H, W) in ((80, 144), (120, 96)):
        stub = types.SimpleNamespace(_y_patch_h=20, _y_patch_w=24, _input_dim_h=H, _input_dim_w=W)
        out["full_%dx%d" % (H, W)] = fn(stub)  # (1, h, w, P) float32
    rng = np.random.default_rng(7)
    for (H, W) in ((320, 1224), (320, 960)):
        stub = types.SimpleNamespace(_y_patch_h=20, _y_patch_w=24, _input_dim_h=H, _input_dim_w=W)
        m = fn(stub)[0]
        h, w, P = m.shape
        n = 4096
        ii, jj, pp = rng.integers(0, h, n), rng.integers(0, w, n), rng.integers(0, P, n)
        out["idx_%dx%d" % (H, W)] = np.stack([pp, ii, jj], 1).astype(np.int32)
        out["val_%dx%d" % (H, W)] = m[ii, jj, pp]
        out["argmax_%dx%d" % (H, W)] = m.reshape(h * w, P).argmax(0).astype(np.int64)
        out["shape_%dx%d" % (H, W)] = np.array(m.shape)
    np.savez_compressed(os.path.join(OUT, "mask_golden.npz"), **out)


def make_msssim():
    sys.modules.setdefault("tensorflow", types.ModuleType("tensorflow"))
    sys.path.insert(0, REF)
    import ms_ssim_np_imgcomp as ref
    rng = np.random.default_rng(11)
    out = {}
    from scipy.ndimage import gaussian_filter
    for k, (H, W) in enumerate(((176, 208), (192, 256))):
        img = gaussian_filter(rng.uniform(0, 255, (H, W, 3)), (3, 3, 0))
        img = np.clip(255 * (img - img.min()) / (img.max() - img.min()), 0, 255).astype(np.uint8)
        rec8 = np.clip(np.round(img.astype(np.float32) + rng.normal(0, 4 + 4 * k, img.shape)), 0, 255).astype(np.uint8)
        rec = rec8.astype(np.float32)  # reconstructions are float arrays in utils.py
        out["img_%d" % k], out["rec_%d" % k] = img, rec8
        out["std_%d" % k] = np.float32(ref._calc_msssim_orig(img[None], rec[None]))
        # utils.msssim_x_vs_rec form: (H,W,3,1)
        out["utils_%d" % k] = np.float32(ref._calc_msssim_orig(img[..., None], rec[..., None]))
    np.savez_compressed(os.path.join(OUT, "msssim_golden.npz"), **out)


def _extract(path, names):
    """Compile the named functions / methods of a reference file in isolation (no module import)."""
    import contextlib
    import functools
    import itertools
    tree = ast.parse(open(os.path.join(REF, path)).read())
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
    for n in body:
        n.decorator_list = []  # staticmethod / property decorators are meaningless outside the class
    tf_stub = types.SimpleNamespace(name_scope=lambda *_a, **_k: contextlib.nullcontext(), Variable=type(None))
    ns = {"np": np, "tf": tf_stub, "functools": functools, "itertools": itertools,
          "_Network3D": types.SimpleNamespace(_make_tf_conv3d_mask=lambda m: m)}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


def make_model_pieces():
    pc = _extract("probclass_imgcomp.py", {
        "create_first_mask", "create_other_mask", "pad_for_probclass3d", "undo_pad_for_probclass3d", "get_np_pad_fn",
        "add_batch_dim", "remove_batch_dim", "_get_ndims", "iter_over_blocks", "num_blocks", "_iter_block_idices",
        "context_shape_from_context_size", "context_size_from_context_shape"})
    out = {}
    net = types.SimpleNamespace(config=types.SimpleNamespace(kernel_size=3), filter_shape=(2, 3, 3))
    out["first_mask"] = pc["create_first_mask"](net)    # (2,3,3,1,1)
    out["other_mask"] = pc["create_other_mask"](net)
    rng = np.random.default_rng(5)
    vol = rng.normal(size=(2, 3, 4, 5)).astype(np.float32)             # NCHW
    out["pad_in"] = vol
    out["pad_out_cs9"] = pc["pad_for_probclass3d"](vol, 9, 1.5)
    out["pad_out_chw_cs5"] = pc["pad_for_probclass3d"](vol[0], 5, -0.25)
    out["unpad_cs9"] = pc["undo_pad_for_probclass3d"](out["pad_out_cs9"][0], 9)  # CHW numpy branch
    out["context_shape_9"] = np.array(pc["context_shape_from_context_size"](9))
    syms = np.arange(4 * 5 * 6).reshape(4, 5, 6)
    blocks = list(pc["iter_over_blocks"](syms, (2, 3, 3)))
    out["block_first_elems"] = np.array([b[0, 0, 0] for b in blocks])
    out["block_count"] = np.array(pc["num_blocks"](syms.shape, (2, 3, 3)))
    ae = _extract("AE.py", {"normalize", "denormalize", "get_mean_var"})
    stub = types.SimpleNamespace(ae_config=types.SimpleNamespace(normalization="FIXED"), get_mean_var=ae["get_mean_var"])
    img = rng.integers(0, 256, size=(2, 3, 6, 7)).astype(np.float32)
    out["norm_in"] = img
    out["norm_out"] = ae["normalize"](stub, img)
    out["denorm_out"] = ae["denormalize"](stub, out["norm_out"])
    mean, var = ae["get_mean_var"]()
    out["mean"], out["var"] = mean, var
    # host-side helpers: pair-list reader (src/DataProvider.py:96-100), L1 metric and PNG writer (src/utils.py:82-111)
    import tempfile
    from PIL import Image
    dp = _extract("DataProvider.py", {"readfiles"})
    ut = _extract("utils.py", {"l1_x_vs_rec", "save_test_imgs_fn"})
    ut["os"], ut["Image"] = os, Image
    with tempfile.TemporaryDirectory() as tmp:
        lst = os.path.join(tmp, "pairs.txt")
        with open(lst, "w") as f:
            f.write("a/image_2/000000_10.png\na/image_3/000000_10.png\n  b/x.png  \nb/y.png\n")
        out["readfiles"] = np.array(dp["readfiles"](types.SimpleNamespace(root_data="/data/"), lst))
        rec = rng.uniform(-3, 260, size=(3, 5, 8)).astype(np.float32).clip(0, 255)
        ut["save_test_imgs_fn"](tmp + "/", "model", rec, 7, 0.0312345)
        name = os.listdir(os.path.join(tmp, "model"))
        out["png_name"] = np.array(name)
        out["png_in"] = rec
        out["png_pixels"] = np.asarray(Image.open(os.path.join(tmp, "model", name[0])))
    a = rng.integers(0, 256, size=(6, 7, 3)).astype(np.uint8)
    b = rng.uniform(0, 255, size=(6, 7, 3)).astype(np.float32)
    diff, l1 = ut["l1_x_vs_rec"](a, b)
    out["l1_a"], out["l1_b"], out["l1_diff"], out["l1_value"] = a, b, diff, np.float32(l1)
    np.savez_compressed(os.path.join(OUT, "model_pieces_golden.npz"), **out)


# ------------------------------------------------------------------------------------------------------------------
# numpy stand-in for the elementwise / shape TensorFlow ops the extracted functions use
# ------------------------------------------------------------------------------------------------------------------
class _Shape(tuple):
    @property
    def ndims(self):
        return len(self)

    def as_list(self):
        return list(self)


class _DType(object):
    def __init__(self, np_dtype):
        self.np_dtype = np.dtype(np_dtype)

    def is_compatible_with(self, other):
        return np.dtype(getattr(other, "np_dtype", other)) == self.np_dtype


def _raw(v):
    return v.a if isinstance(v, _T) else v


class _T(object):
    """A 'tensor': numpy array + the attribute surface the reference code touches."""

    def __init__(self, a):
        self.a = np.asarray(_raw(a))

    shape = property(lambda self: _Shape(self.a.shape))
    dtype = property(lambda self: _DType(self.a.dtype))

    def get_shape(self):
        return self.shape

    def __getitem__(self, idx):
        return _T(self.a[idx])

    def __len__(self):
        return len(self.a)

    def __int__(self):
        return int(self.a)

    def __index__(self):
        return int(self.a)

    def __format__(self, spec):
        return format(str(self.a.shape), spec)


for _name, _fn in (("add", np.add), ("sub", np.subtract), ("mul", np.multiply), ("truediv", np.true_divide)):
    setattr(_T, "__%s__" % _name, (lambda f: lambda self, o: _T(f(self.a, _raw(o))))(_fn))
    setattr(_T, "__r%s__" % _name, (lambda f: lambda self, o: _T(f(_raw(o), self.a)))(_fn))
_T.__neg__ = lambda self: _T(-self.a)


def _softmax(v, axis=-1):
    a = _raw(v)
    e = np.exp(a - a.max(axis=axis, keepdims=True))
    return _T((e / e.sum(axis=axis, keepdims=True)).astype(a.dtype))


def _one_hot(idx, depth, axis=-1, dtype=None):
    i = _raw(idx)
    return _T((np.arange(depth) == i[..., None]).astype(np.float32))


def _make_tf():
    import contextlib
    f32 = np.float32
    nn = types.SimpleNamespace(sigmoid=lambda v: _T((f32(1) / (f32(1) + np.exp(-_raw(v)))).astype(f32)), softmax=_softmax)
    return types.SimpleNamespace(
        float32=_DType(np.float32), nn=nn, name_scope=lambda *_a, **_k: contextlib.nullcontext(),
        tile=lambda v, reps: _T(np.tile(np.asarray(_raw(v), dtype=np.float32), reps)),
        expand_dims=lambda v, axis: _T(np.expand_dims(_raw(v), axis)),
        divide=lambda a, b: _T(np.true_divide(_raw(a), _raw(b))),
        split=lambda v, sizes, axis: [_T(p) for p in np.split(_raw(v), np.cumsum(sizes)[:-1], axis=axis)],
        concat=lambda vs, axis: _T(np.concatenate([_raw(v) for v in vs], axis=axis)),
        clip_by_value=lambda v, lo, hi: _T(np.clip(_raw(v), lo, hi)),
        range=lambda n, dtype=None: _T(np.arange(n, dtype=np.float32)),
        reshape=lambda v, shp: _T(np.reshape(_raw(v), [int(_raw(s_)) for s_ in _raw(shp)])),
        maximum=lambda a, b, name=None: _T(np.maximum(_raw(a), _raw(b)).astype(np.float32)),
        minimum=lambda a, b, name=None: _T(np.minimum(_raw(a), _raw(b)).astype(np.float32)),
        shape=lambda v: _T(np.array(_raw(v).shape, dtype=np.int32)),
        square=lambda v: _T(np.square(_raw(v))), abs=lambda v: _T(np.abs(_raw(v))),
        argmax=lambda v, axis: _T(np.argmax(_raw(v), axis=axis).astype(np.int64)),
        one_hot=_one_hot,
        reduce_sum=lambda v, axis=None, name=None: _T(np.sum(_raw(v), axis=axis, dtype=np.float32)),
        reduce_prod=lambda v: _T(np.prod(_raw(v))),
        to_float=lambda v: _T(np.float32(_raw(v))),
        int32=_DType(np.int32),
        cast=lambda v, dt: _T(np.asarray(_raw(v)).astype(dt.np_dtype)),  # float -> int32 truncates toward zero, as TF
        constant=lambda v, dtype=None, name=None: _T(np.asarray(v, dtype=(dtype.np_dtype if dtype else None))),
        reduce_mean=lambda v, axis=None, name=None: _T(np.mean(np.asarray(_raw(v)), dtype=np.float32,
                                                               axis=(tuple(axis) if isinstance(axis, list) else axis))),
    )


def _extract_tf(path, names, consts=()):
    """Like _extract, for functions that call tf ops: runs them against the numpy stand-in."""
    tree = ast.parse(open(os.path.join(REF, path)).read())
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
    body += [n for n in tree.body if isinstance(n, ast.Assign) and any(getattr(t, "id", None) in consts for t in n.targets)]
    for n in body:
        if isinstance(n, ast.FunctionDef):
            n.decorator_list = []
    ns = {"np": np, "tf": _make_tf()}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


def make_tf_pieces():
    rng = np.random.default_rng(23)
    out = {}
    cfg = types.SimpleNamespace(use_L2andLAB=False)
    sf = _extract_tf("siFinder.py", {"reduce_mean_and_std_normalize_images", "rgb_transform"})
    img = rng.integers(0, 256, size=(5, 20, 24, 3)).astype(np.float32)  # patches, channel last
    out["sif_in"] = img
    norm = sf["reduce_mean_and_std_normalize_images"](_T(img), cfg)
    out["sif_norm"] = norm.a
    out["sif_rgb"] = sf["rgb_transform"](norm, cfg).a
    ae = _extract_tf("autoencoder_imgcomp.py", {"_get_heatmap3D", "_mask_with_heatmap"})
    z33 = (1.5 * rng.standard_normal((2, 33, 6, 7))).astype(np.float32)
    z33[0, 0, :2] = -30.0
    z33[1, 0, 2:4] = 30.0
    out["z33"] = z33
    hm = ae["_get_heatmap3D"](_T(z33))
    out["heatmap3d"] = hm.a
    out["z_masked"] = ae["_mask_with_heatmap"](_T(z33), hm).a
    qz = _extract_tf("quantizer_imgcomp.py", {"_quantize1d", "phi_times_centers"}, consts=("_HARD_SIGMA",))
    centers = np.array([0.55, -0.92, -1.84, -1.93, 1.25, 1.65], dtype=np.float32)
    x = out["z_masked"].copy()
    x[0, 0, 0, :6] = centers          # exactly on a centre
    x[0, 1, 0, 0] = np.float32(0.5 * (centers[2] + centers[3]))  # midway between the two closest centres
    out["q_in"], out["q_centers"] = x, centers
    qsoft, qhard, sym = qz["_quantize1d"](_T(x), _T(centers), 1, "NCHW")
    out["q_soft"], out["q_hard"], out["q_symbols"] = qsoft.a, qhard.a, sym.a
    bits = _extract_tf("bits_imgcomp.py", {"bitcost_to_bpp", "num_pixels_in_input_batch"})
    bc = rng.uniform(0, 4, size=(2, 32, 5, 9)).astype(np.float32)
    inp = np.zeros((2, 3, 40, 72), np.float32)
    out["bc"], out["bc_input_shape"] = bc, np.array(inp.shape)
    out["bpp"] = np.float32(bits["bitcost_to_bpp"](_T(bc), _T(inp)).a)
    np.savez_compressed(os.path.join(OUT, "tf_pieces_golden.npz"), **out)


def make_loss_pieces():
    """The loss arithmetic of siNet_validate (src/AE.py:76-99): the reference's own Distortions class and get_loss
    (src/Distortions_imgcomp.py:7-56,68-146) executed on the numpy stand-in, for all three restated distortions."""
    tree = ast.parse(open(os.path.join(REF, "Distortions_imgcomp.py")).read())
    body = [n for n in tree.body if (isinstance(n, ast.ClassDef) and n.name == "Distortions")
            or (isinstance(n, ast.FunctionDef) and n.name == "get_loss")]
    tf = _make_tf()
    helpers = types.SimpleNamespace(  # fjcommon.tf_helpers.log10: log(x) / log(10)
        log10=lambda v: _T((np.log(_raw(v)) / np.float32(np.log(10.0))).astype(np.float32)),
        list_without_None=lambda *a: [v for v in a if v is not None])
    ns = {"np": np, "tf": tf, "tf_helpers": helpers}
    exec(compile(ast.Module(body=body, type_ignores=[]), "Distortions_imgcomp.py", "exec"), ns)
    rng = np.random.default_rng(31)
    out = {}
    x = rng.integers(0, 256, size=(3, 3, 16, 24)).astype(np.float32)
    x_out = np.clip(x + 6.0 * rng.standard_normal(x.shape), 0, 255).astype(np.float32)
    bc = rng.uniform(0, 4, size=(3, 32, 2, 3)).astype(np.float32)
    hm = np.clip(rng.uniform(-0.5, 1.5, size=bc.shape), 0, 1).astype(np.float32)
    out["x"], out["x_out"], out["bc"], out["heatmap"] = x, x_out, bc, hm
    regs = {"enc": np.float32(0.375), "dec": np.float32(0.125)}
    ae = types.SimpleNamespace(encoder_regularization_loss=lambda: _T(regs["enc"]),
                               decoder_regularization_loss=lambda: _T(regs["dec"]))
    pc = types.SimpleNamespace(regularization_loss=lambda: None)
    for name in ("mae", "mse", "psnr"):
        for h_target in (0.04, 2.5):  # the rate term active / clamped at zero
            cfg = types.SimpleNamespace(distortion_to_minimize=name, K_psnr=100, K_ms_ssim=5000, H_target=h_target, beta=500)
            d = ns["Distortions"](cfg, _T(x), _T(x_out), is_training=True)
            out["d_%s" % name] = np.float32(d.d_loss_scaled.a)
            total, h_real, pc_comps, _ae_comps = ns["get_loss"](cfg, ae, pc, _T(np.float32(0.3)) * d.d_loss_scaled, _T(bc), _T(hm))
            out["total_%s_%g" % (name, h_target)] = np.float32(total.a)
            out["H_real"] = np.float32(h_real.a)
            out["H_mask"] = np.float32(dict(pc_comps)["H_mask"].a)
    out["reg_enc"], out["reg_dec"] = regs["enc"], regs["dec"]
    np.savez_compressed(os.path.join(OUT, "loss_pieces_golden.npz"), **out)


def make_configs():
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from dsin_b200 import config_parser
    out = {}
    for name in ("ae_run_configs", "pc_run_configs"):
        cfg, _ = config_parser.parse(os.path.join(REF, "run_configs", name))
        out[name] = {k: repr(v) for k, v in cfg.all_params_and_values()}
    with open(os.path.join(OUT, "run_configs_golden.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    REF = os.path.join(sys.argv[1], "src")
    make_configs()
    make_loss_pieces()
    make_masks()
    make_msssim()
    make_model_pieces()
    make_tf_pieces()
    for f in ("mask_golden.npz", "msssim_golden.npz", "model_pieces_golden.npz", "tf_pieces_golden.npz",
              "loss_pieces_golden.npz", "run_configs_golden.json"):
        print(f, os.path.getsize(os.path.join(OUT, f)))
