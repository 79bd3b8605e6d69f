"""Host-side logic that runs without a GPU: config parser, synthetic generators, weight naming."""
import json
import os

import numpy as np
import pytest
import torch

from dsin_b200 import config_parser, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_parse_shipped_configs():
    ae, rel = config_parser.parse(os.path.join(ROOT, "dsin_b200", "run_configs", "ae_run_configs"))
    pc, _ = config_parser.parse(os.path.join(ROOT, "dsin_b200", "run_configs", "pc_run_configs"))
    assert rel == "ae_run_configs"
    assert ae.crop_size == (320, 1224) and ae.y_patch_size == (20, 24) and ae.batch_size == 1
    assert ae.H_target == pytest.approx(0.04) and ae.normalization == "FIXED" and ae.distortion_to_minimize == "mae"
    assert ae.arch == "CVPR" and ae.arch_param_B == 5 and ae.num_chan_bn == 32 and ae.num_centers == 6
    assert ae.AE_only is False and ae.use_gauss_mask is True and ae.lr_centers_factor is None
    assert pc.arch == "res_shallow" and pc.kernel_size == 3 and pc.arch_param__k == 24
    assert pc.use_centers_for_padding is True and pc.regularization_factor is None


def test_parse_reference_config_files_verbatim(golden_dir):
    """The shipped run configs parse to exactly what the reference's src/run_configs parse to (repr of every value,
    stored by tests/golden/make_golden.py)."""
    with open(os.path.join(golden_dir, "run_configs_golden.json")) as f:
        ref = json.load(f)
    for name in ("ae_run_configs", "pc_run_configs"):
        mine, _ = config_parser.parse(os.path.join(ROOT, "dsin_b200", "run_configs", name))
        assert {k: repr(v) for k, v in mine.all_params_and_values()} == ref[name]


def test_constraint_violation_and_bad_lines():
    with pytest.raises(ValueError):
        config_parser.parse_string("constrain opt :: A, B\nopt = C\n")
    with pytest.raises(ValueError):
        config_parser.parse_string("this is not a config line\n")
    cfg = config_parser.parse_string("a = 2*3  # trailing\nb = (a, 'x#y')\n")
    assert cfg.a == 6 and cfg.b == (6, "x#y")


def test_weight_names_and_shapes():
    W = synth.make_weights(0)
    assert W[synth.ENC + "h1/weights"].shape == (5, 5, 3, 64)
    assert W[synth.ENC + "to_bn/weights"].shape == (5, 5, 128, 33)
    assert W[synth.ENC + "res_block_enc_4/enc_4_3/conv2/weights"].shape == (3, 3, 128, 128)
    assert W[synth.DEC + "from_bn/weights"].shape == (3, 3, 128, 32)
    assert W[synth.DEC + "h13/weights"].shape == (5, 5, 3, 64)
    assert W[synth.PC + "res1/conv3d_conv1_mask/weights"].shape == (2, 3, 3, 24, 24)
    assert W[synth.SIN + "g_conv1/weights"].shape == (3, 3, 6, 32)
    assert W[synth.SIN + "g_conv_last/weights"].shape == (1, 1, 32, 3)
    n_ae = sum(v.size for k, v in W.items() if k.endswith("/weights") and ("encoder" in k or k.startswith("decoder")))
    assert 9.9e6 < n_ae < 10.2e6  # SURVEY App. A.11: ~10.0 M conv parameters
    assert len(synth.enc_conv_scopes()) == 34 and len(synth.dec_conv_scopes()) == 32


def test_weights_roundtrip(tmp_path):
    W = synth.make_weights(1)
    p = str(tmp_path / "w.npz")
    synth.save_weights(p, W)
    W2 = synth.load_weights(p)
    assert sorted(W) == sorted(W2)
    assert all(np.array_equal(W[k], W2[k]) for k in W)


def test_synthetic_pairs_are_seeded_and_uint8_valued():
    x1, y1 = synth.make_pair(5, 80, 144)
    x2, y2 = synth.make_pair(5, 80, 144)
    assert np.array_equal(x1, x2) and np.array_equal(y1, y2)
    assert x1.shape == (3, 80, 144) and x1.dtype == np.float32
    assert np.array_equal(x1, np.floor(x1)) and x1.min() >= 0 and x1.max() <= 255
    xs, ys = synth.make_batch(3, 40, 48, seed=9)
    assert xs.shape == (3, 3, 40, 48) and ys.shape == xs.shape


def test_bitstream_container_roundtrip():
    from dsin_b200 import bitstream
    streams = [b"", b"\x01\x02\x03", bytes(range(200)), b"\xff"]
    blob = bitstream.pack(streams, 32, 40, 153, 6)
    assert blob[:4] == b"DSPC" and len(blob) == 16 + 4 * 4 + sum(map(len, streams))
    assert bitstream.unpack(blob) == (32, 40, 153, 6, streams)
    assert bitstream.payload_bits(blob) == 8 * 204
    import pytest as _pt
    for bad in (blob[:10], blob[:-1], blob + b"\x00", b"DSPX" + blob[4:], blob[:4] + b"\x09" + blob[5:]):
        with _pt.raises(ValueError):
            bitstream.unpack(bad)


def test_config_values_are_evaluated_without_eval():
    """Arithmetic, tuples, earlier keys and constraint words work; attribute walks, calls and subscripts do not."""
    from dsin_b200 import config_parser
    cfg = config_parser.parse_string("a = 2*0.02\nb = (320, 1224)\nc = a * 3 + 1\nconstrain n :: OFF, FIXED\nn = FIXED\nd = -2**3")
    assert cfg.a == 0.04 and cfg.b == (320, 1224) and cfg.c == 0.04 * 3 + 1 and cfg.n == "FIXED" and cfg.d == -8
    for bad in ("x = ().__class__", "x = open('f')", "x = [1][0]", "x = (1).real", "x = 9**9**9", "x = [i for i in (1,)]"):
        with pytest.raises(ValueError):
            config_parser.parse_string(bad)


def test_bitstream_header_is_validated_before_allocation():
    """A foreign / malformed container must be refused from its header alone (no device work, no big allocation)."""
    from dsin_b200 import bitstream
    from dsin_b200.probclass_imgcomp import _ResShallow
    blob = bitstream.pack([b"\x00" * 4] * 8, 65535, 65535, 65535, 6)
    pc = _ResShallow.__new__(_ResShallow)
    pc.L = 6
    pc.config = type("C", (), {"use_centers_for_padding": True, "arch_param__k": 24})()
    with pytest.raises(ValueError, match="symbol volume|outside"):
        pc.decode_symbols([blob], None, expect_shape=(32, 40, 153))
    with pytest.raises(ValueError, match="outside"):
        pc.decode_symbols([blob], None)
    ok = bitstream.pack([b"\x00" * 70000] + [b"\x00"] * 7, 32, 40, 153, 6)
    with pytest.raises(ValueError, match="longer than"):
        pc.decode_symbols([ok], None, expect_shape=(32, 40, 153))


def test_host_staging_copy_matches_numpy_assignment():
    """AE._host_copy: the 8-byte-word fast path (torch's threaded copy) and the numpy fallback give the same bytes, for
    whole buffers and for the per-chunk slices the pipelined entry point stages."""
    from dsin_b200.AE import _host_copy
    rng = np.random.default_rng(9)
    old = torch.get_num_threads()
    try:
        for threads in (1, 2):
            torch.set_num_threads(threads)
            for shape, dt in (((16, 3, 320, 1224), np.uint8), ((3, 3, 37, 41), np.uint8), ((8, 3, 80, 144), np.float32)):
                a = rng.integers(0, 256, size=shape).astype(dt)
                dst = torch.zeros(shape, dtype=torch.from_numpy(a[:0]).dtype)
                _host_copy(dst, a)
                assert np.array_equal(dst.numpy(), a)
                if shape[0] % 2 == 0:
                    dst.zero_()
                    h = shape[0] // 2
                    for sl in (slice(0, h), slice(h, shape[0])):
                        _host_copy(dst[sl], a[sl])
                    assert np.array_equal(dst.numpy(), a)
    finally:
        torch.set_num_threads(old)


def test_main_parser_has_the_validation_step_switch():
    from dsin_b200 import main as dmain
    a = dmain.build_parser().parse_args(["--validate", "--synthetic", "2", "--no_save_test_img"])
    assert a.validate and a.synthetic == 2 and a.no_save_test_img
    assert not dmain.build_parser().parse_args([]).validate
