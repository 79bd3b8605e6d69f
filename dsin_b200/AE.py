"""AE facade (/root/reference/src/AE.py) on libdsin_b200: same constructor and inference methods.

    AE(ae_config, pc_config, encoder, decoder, siFinder, SI_full_img, siNet, cur_dir)
    siNet_get_reconstructed(x, y) -> (y_dec, y_syn, x_dec, x_with_si, bpp)     src/AE.py:132-148
    siNet_validate(x, y) -> loss_test (forward pass + loss reductions)         src/AE.py:76-99,120-131
    create_y_dec(y)                                                            src/AE.py:150-152
    load_model(path) / save_model(path)                                        src/AE.py:154-175

Differences (documented in DESIGN.md): inputs may hold B >= 1 pairs (the reference's SI path is
hard-wired to batch 1, src/AE.py:26) -- each pair is processed with batch-1 semantics and bpp is
the batch aggregate of bits.bitcost_to_bpp; the two autoencoder passes (on y and on x) run as
one batch of 2B images; weights are read from a TF-V2 checkpoint (tf_checkpoint.py, no TensorFlow) or an
.npz keyed by the TF variable names; the training step (siNet_update) raises NotImplementedError.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import autoencoder_imgcomp as autoencoder
from . import Distortions_imgcomp as Distortions
from . import bits_imgcomp as bits
from . import ops
from . import precision as precision_policy
from . import probclass_imgcomp as probclass
from . import synth
from . import tf_checkpoint
from .siFinder import GaussianPrior, uses_l2


def _host_copy(dst, a):
    """Contiguous numpy array -> pinned tensor of the same shape and dtype.  Copied as 8-byte words by torch's
    multi-threaded copy when the size allows (a 1-byte-element copy_ is not vectorised, and numpy's assignment is one
    memcpy thread: 75 MB of uint8 images per micro-batch of 32 pairs took 5 ms of the end-to-end call)."""
    if a.nbytes >= (1 << 20) and a.nbytes % 8 == 0 and torch.get_num_threads() > 1:
        dst.view(-1).view(torch.int64).copy_(torch.from_numpy(a.reshape(-1).view(np.int64)))
    else:
        dst.numpy()[...] = a


class AE(object):
    def __init__(self, ae_config, pc_config, encoder, decoder, siFinder, SI_full_img, siNet, cur_dir,
                 weights=None, seed=0, device=None, precision=None):
        self.ae_config = ae_config
        self.pc_config = pc_config
        self._encode = encoder
        self._decode = decoder
        self.AE_only = self.ae_config.AE_only
        self.si_weight = 0.0 if self.AE_only else self.ae_config.si_weight
        self._siNet = siNet.clone() if hasattr(siNet, "clone") else siNet
        self._SI_full_img = SI_full_img
        self._siFinder = siFinder
        self.use_y_gauss_mask = self.ae_config.use_gauss_mask
        self._batch_size = self.ae_config.batch_size if self.AE_only else 1
        self._input_dim_h, self._input_dim_w = self.ae_config.crop_size
        self._y_patch_h, self._y_patch_w = self.ae_config.y_patch_size
        try:  # the reference opens the train list at construction (src/AE.py:29); absent at inference
            with open(os.path.join(cur_dir or "", ae_config.file_path_train)) as f:
                self.num_training_imgs = sum(1 for _ in f) // 2
        except (OSError, TypeError):
            self.num_training_imgs = 0
        if getattr(self.ae_config, "normalization", "FIXED") not in ("FIXED",):
            raise ValueError("Invalid normalization style {} (only FIXED is built)".format(
                self.ae_config.normalization))
        if not getattr(self.ae_config, "heatmap", True):
            raise NotImplementedError("heatmap=False is not built")

        # One process drives one GPU (SURVEY 8e): the AE lives on torch's CURRENT device.  `device`, if given, must
        # name that device -- every kernel is launched on the current device's stream and the C library rejects a
        # handle whose device is not current.
        cur = torch.cuda.current_device() if torch.cuda.is_available() else 0
        if device is not None and torch.device("cuda", device if isinstance(device, int) else
                                               torch.device(device).index or 0).index != cur:
            raise ValueError("AE(device=%r): call torch.cuda.set_device() first -- dsin_b200 runs one process per GPU "
                             "on the current CUDA device (cuda:%d)" % (device, cur))
        ops.handle(cur)  # fails loudly without libdsin_b200.so / an sm_100 GPU
        self.device = torch.device("cuda", cur)
        self.precision = precision_policy.get(precision)
        self.ae_imgcomp = autoencoder.get_network_cls(self.ae_config)(self.ae_config)
        self.pc_imgcomp = probclass.get_network_cls(self.pc_config)(self.pc_config,
                                                                    num_centers=self.ae_config.num_centers)
        self.mask = self.create_gaussian_masks() if self.use_y_gauss_mask else 1
        self.weights = None
        self.set_weights(weights if weights is not None else synth.make_weights(seed))
        self._pinned = {}
        self._ring = 0
        self._copy_stream = None
        self._in_stream = None
        self._dev_in = {}
        self.last = {}
        # CUDA graphs for the numpy entry points: one capture per input shape, replayed afterwards, so a call
        # costs two graph launches instead of ~230 kernel launches (batch 1 is launch-bound otherwise)
        self.use_cuda_graph = True  # set to False for eager launches (tests compare the two)
        self.e2e_overlap = True     # copy y_dec/x_dec out on a side stream while the SI-Finder / SI-Net run
        self.e2e_chunk = 8          # numpy calls with more pairs than this run as a pipeline of chunks of this many
        self._graphs = {}

    # ------------------------------------------------------------------ weights
    def set_weights(self, W):
        """W: dict keyed by TF variable names (SURVEY App. A.11)."""
        self.weights = W
        if getattr(self, "_graphs", None):
            self._graphs.clear()  # captured graphs point at the previous weight tensors
        self.ae_imgcomp.load_weights(W)
        self.pc_imgcomp.load_weights(W)
        if not self.AE_only:
            self._siNet.load_weights(W)

    def save_model(self, save_path):
        """src/AE.py:154-156 (`tf.train.Saver.save`): writes a TF-V2 checkpoint `<save_path>.index` +
        `<save_path>.data-00000-of-00001` keyed by the TF variable names; a path ending in .npz writes the
        same dictionary as an .npz instead."""
        if save_path.endswith(".npz"):
            os.makedirs(os.path.dirname(os.path.abspath(save_path)), exist_ok=True)
            synth.save_weights(save_path, self.weights)
        else:
            tf_checkpoint.write_checkpoint(save_path, self.weights)

    def _restore_names(self):
        """The variables `load_model` of the reference restores for inference (src/AE.py:158-172): scopes
        encoder/encoder_body, decoder, imgcomp and -- unless AE_only -- siNetwork.  Optimizer slots and the
        training step of a training checkpoint are ignored."""
        c = self.ae_config
        with_si = (not self.AE_only) and (getattr(c, "load_train_step", False) or
                                          (getattr(c, "test_model", True) and not getattr(c, "train_model", False)))
        names = [k for k in synth.variable_names(c.arch_param_B) if
                 k.startswith(("encoder/encoder_body/", "decoder/", "imgcomp/"))
                 or (with_si and k.startswith("siNetwork/"))]
        return names

    def load_model(self, load_path):
        """Accepts what `tf.train.Saver.restore` takes (a TF-V2 checkpoint prefix, src/AE.py:158-175) or an
        .npz keyed by the same variable names."""
        npz = load_path if load_path.endswith(".npz") else load_path + ".npz"
        if not load_path.endswith(".npz") and tf_checkpoint.checkpoint_exists(load_path):
            print("Loading " + load_path)
            W = tf_checkpoint.read_checkpoint(load_path, names=self._restore_names())
        elif os.path.exists(npz):
            print("Loading " + npz)
            W = synth.load_weights(npz)
        else:
            raise FileNotFoundError("neither {}.index (TF-V2 checkpoint) nor {} found".format(load_path, npz))
        if not self.AE_only and not any(k.startswith("siNetwork/") for k in W):
            # "train SI for the first time from an AE checkpoint" (src/AE.py:163-172): the reference restores the
            # AE scopes only and keeps the SI-Net's initialiser values
            for k, v in self.weights.items():
                if k.startswith("siNetwork/"):
                    W[k] = v
        self.set_weights(W)

    # ------------------------------------------------------------------ helpers kept from the reference
    def create_gaussian_masks(self):
        """The reference returns a (1,h,w,P) float32 constant (1.18 GB at 320x1224); the kernels
        evaluate the same prior analytically, so only its geometry is returned."""
        return GaussianPrior(self._input_dim_h, self._input_dim_w, self._y_patch_h, self._y_patch_w)

    @staticmethod
    def get_mean_var():
        mean = np.array([93.70454143384742, 98.28243432206516, 94.84678088809876], dtype=np.float32)
        var = np.array([5411.79935676, 5758.60456747, 5890.31451232], dtype=np.float32)
        return mean.reshape(3, 1, 1), var.reshape(3, 1, 1)

    def siNet_update(self, x, y):
        raise NotImplementedError("the training step (gradients, optimiser) is not built; dsin_b200 has the forward "
                                  "passes only: siNet_get_reconstructed and siNet_validate")

    def siNet_validate(self, x, y):
        """x, y: (B,3,H,W) uint8 / uint8-valued arrays -> the scalar validation loss `loss_test` of src/AE.py:120-131:
        one forward pass in inference mode, then
            (1 - si_weight) * d_loss_scaled(x, x_dec) + beta * max(H_soft - H_target, 0) + reg
            + si_weight * mean|x - x_with_si|                      (src/AE.py:76-99, src/Distortions_imgcomp.py:113-146).
        The forward pass is the one siNet_get_reconstructed runs (same kernels, same CUDA graphs); the reductions are
        one more launch pair (csrc/loss.cu).  The components are kept in `self.last_loss`."""
        xs, ys = self._stage(x, "x"), self._stage(y, "y")
        if self.use_cuda_graph:
            out = self.replay_device(xs, ys)
            xd = self._graph_state(xs.shape[0], xs.shape[2], xs.shape[3])["x"]
        else:
            xd = xs.to(torch.float32)
            out = self.reconstruct_device(xd, ys.to(torch.float32))
        self.last = out
        loss, comps = self.validation_loss_device(xd, out)
        self.last_loss = comps
        return loss

    def validation_loss_device(self, x, out):
        """x (B,3,H,W) fp32 CUDA tensor and the dict reconstruct_device / replay_device returned for it ->
        (loss_test, components)."""
        c = self.ae_config
        terms = ops.validation_terms(x, out["x_dec"].contiguous(), None if self.AE_only else out["x_with_si"],
                                     out["bits"], out["heatmap"], squared=Distortions.squared_distortion(c))
        t = terms.cpu().numpy()  # (B, 4) float64 per-image sums; synchronises the stream
        B = x.shape[0]
        img_elems, sym_elems = x.numel() // B, out["bits"].numel() // B
        d = Distortions.distortion_to_minimize(c, t[:, 0], img_elems)
        H_real = np.float32(t[:, 2].sum() / float(B * sym_elems))
        H_mask = np.float32(t[:, 3].sum() / float(B * sym_elems))
        w = np.float32(self.si_weight)
        total, H_real, pc_comps, ae_comps = Distortions.get_loss(c, self.ae_imgcomp, self.pc_imgcomp,
                                                                 np.float32(np.float32(1) - w) * d, H_real, H_mask)
        # tf.losses.absolute_difference: sum of |x - x_with_si| over the number of elements (src/AE.py:94)
        loss_siNet = np.float32(0) if self.AE_only else np.float32(t[:, 1].sum() / float(B * img_elems))
        loss_test = np.float32(total + np.float32(w * loss_siNet))
        comps = dict(pc_comps + ae_comps)
        comps.update({"d_loss": d, "total_loss_test": total, "loss_siNet": loss_siNet, "loss_test": loss_test})
        return float(loss_test), comps

    # ------------------------------------------------------------------ host <-> device staging
    def _stage(self, a, slot):
        """Host array / tensor -> device tensor in its own dtype (uint8 images travel as uint8)."""
        if torch.is_tensor(a):
            return a.contiguous() if a.is_cuda else a.to(self.device, non_blocking=True)
        a = np.ascontiguousarray(a)
        key = (slot, a.shape, a.dtype.str)
        buf = self._pinned.get(key)
        if buf is None:
            buf = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
            self._pinned[key] = buf
        _host_copy(buf, a)
        return buf.to(self.device, non_blocking=True)

    def _to_device(self, a, slot):
        return self._stage(a, slot).to(torch.float32)

    def pinned_like(self, shape, dtype=np.float32):
        """A pinned host tensor callers can fill in place and pass to siNet_get_reconstructed."""
        return torch.empty(tuple(shape), dtype=torch.from_numpy(np.zeros(0, dtype)).dtype, pin_memory=True)

    def _to_host(self, tensors):
        self._ring ^= 1
        outs = []
        for i, t in enumerate(tensors):
            key = ("out", i, self._ring, tuple(t.shape))
            buf = self._pinned.get(key)
            if buf is None:
                buf = torch.empty(tuple(t.shape), dtype=t.dtype, pin_memory=True)
                self._pinned[key] = buf
            buf.copy_(t, non_blocking=True)
            outs.append(buf)
        torch.cuda.current_stream().synchronize()
        return [b.numpy() for b in outs]

    # ------------------------------------------------------------------ inference
    def reconstruct_device(self, x, y, on_decoded=None, on_found=None):
        """Device-resident variant: x, y (B,3,H,W) fp32 CUDA tensors -> dict of CUDA tensors.
        on_decoded(dec) is called as soon as the decoder output (2B,3,H,W) = [y_dec; x_dec] is enqueued and
        on_found(y_syn) as soon as the SI-Finder's output is, so a caller can start copying them out while the
        SI-Finder resp. the SI-Net run."""
        out = self._encode_decode(x, y)
        if on_decoded is not None:
            on_decoded(out["dec"])
        out.update(self._find_side_information(out["dec"], y, x.shape[0]))
        if on_found is not None:
            on_found(out["y_syn"])
        out.update(self._fuse_side_information(out))
        return out

    def _encode_decode(self, x, y):
        """AE(y) and AE(x) as one batch of 2B images (src/AE.py:50-57,150-152) + bit cost of x (src/AE.py:85-87)."""
        B = x.shape[0]
        P = self.precision
        if P.enc_x == P.enc_y:
            z = self._encode(torch.cat([y, x], dim=0), self.ae_imgcomp, is_training=False, terms=P.enc_x)
            qall, qx, sx, sy, hx = z.qbar, z.qbar[B:], z.symbols[B:], z.symbols[:B], z.heatmap[B:]
        else:  # the two encoder passes run at different operand precision: two launches per layer
            zy = self._encode(y, self.ae_imgcomp, is_training=False, terms=P.enc_y)
            zx = self._encode(x, self.ae_imgcomp, is_training=False, terms=P.enc_x)
            qall, qx, sx, sy, hx = self._cat_qbar(zy.qbar, zx.qbar), zx.qbar, zx.symbols, zy.symbols, zx.heatmap
        dec = self._decode(qall, self.ae_imgcomp, is_training=False, terms=P.dec)
        bc = self.pc_imgcomp.bitcost(qx, sx, is_training=False,
                                     pad_value=self.pc_imgcomp.auto_pad_value(self.ae_imgcomp), terms=P.probclass)
        return {"dec": dec, "symbols": sx, "symbols_y": sy, "qbar": qx, "bits": bc, "bits_sum": bc._dsin_sum,
                "heatmap": hx}

    @staticmethod
    def _cat_qbar(qa, qb):
        """Concatenate two bottlenecks along the batch, keeping the NHWC twin the decoder consumes."""
        q = torch.cat([qa, qb], dim=0)
        na, nb = getattr(qa, "_dsin_nhwc", None), getattr(qb, "_dsin_nhwc", None)
        if na is not None and nb is not None:
            q._dsin_nhwc = torch.cat([na, nb], dim=0)
        return q

    def replay_device(self, x, y):
        """reconstruct_device through the captured CUDA graphs: x, y (B,3,H,W) CUDA tensors (any dtype) are copied
        into the captured input buffers, the three graphs are replayed, and the dict of STATIC output tensors is
        returned (overwritten by the next replay)."""
        st = self._graph_state(x.shape[0], x.shape[2], x.shape[3])
        st["x"].copy_(x)
        st["y"].copy_(y)
        st["g_head"].replay()
        st["g_find"].replay()
        st["g_net"].replay()
        return dict(st["out"])

    def _graph_state(self, B, H, W):
        """Capture (once per shape) the three segments of the inference step -- AE(y) + AE(x) + bit cost, SI-Finder,
        SI-Net -- as CUDA graphs over static buffers (segments, so that each segment's outputs can be copied to the host
        while the next one runs).  The SI-Finder's matching mode is part of the key: switching ae_config.use_L2andLAB
        on a live AE captures the other mode's graphs instead of replaying these."""
        key = (B, H, W, uses_l2(self.ae_config))
        st = self._graphs.get(key)
        if st is not None:
            return st
        x = torch.zeros((B, 3, H, W), dtype=torch.float32, device=self.device)
        y = torch.zeros_like(x)
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):  # warm-up: one-time allocations and kernel attributes happen here
            for _ in range(2):
                self.reconstruct_device(x, y)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        g_head, g_find, g_net = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_head, capture_error_mode="thread_local"):
            out = self._encode_decode(x, y)
        with torch.cuda.graph(g_find, pool=g_head.pool(), capture_error_mode="thread_local"):
            out.update(self._find_side_information(out["dec"], y, B))
        with torch.cuda.graph(g_net, pool=g_head.pool(), capture_error_mode="thread_local"):
            out.update(self._fuse_side_information(out))
        st = {"x": x, "y": y, "g_head": g_head, "g_find": g_find, "g_net": g_net, "out": out}
        self._graphs[key] = st
        return st

    def decode_side_device(self, qbar_x, y):
        """Receiver side only (SURVEY 8d "decode-side" region): the quantised bottleneck of x (what the
        bitstream carries) and the side image y -> AE(y) (src/AE.py:150-152), decoder(x) (src/AE.py:57),
        SI-Finder and SI-Net (src/AE.py:60-69).  No encoder pass over x and no probability model."""
        B = y.shape[0]
        zy = self._encode(y, self.ae_imgcomp, is_training=False, terms=self.precision.enc_y)
        dec = self._decode(torch.cat([zy.qbar, qbar_x], dim=0), self.ae_imgcomp, is_training=False,
                           terms=self.precision.dec)
        return self._side_information(dec, y, B)

    def _side_information(self, dec, y, B):
        out = self._find_side_information(dec, y, B)
        out.update(self._fuse_side_information(out))
        return out

    def _find_side_information(self, dec, y, B):
        """SI-Finder (src/AE.py:58-61): y_syn = the side image re-assembled from the best-matching patches."""
        dec_nhwc = dec._dsin_nhwc
        y_dec, x_dec = dec[:B], dec[B:]
        y_dec._dsin_nhwc, x_dec._dsin_nhwc = dec_nhwc[:B], dec_nhwc[B:]
        out = {"y_dec": y_dec, "x_dec": x_dec}
        if self.AE_only:
            out["y_syn"] = torch.zeros_like(y)
            return out
        y_syn, _ncc, _arg, _q, _r, row, col, _xp, _yp = self._SI_full_img(
            x_dec, y, self.mask, self._y_patch_h, self._y_patch_w, self.ae_config, y_dec)
        out.update({"y_syn": y_syn, "row": row, "col": col, "best": getattr(y_syn, "_dsin_best", None)})
        return out

    def _fuse_side_information(self, found):
        """SI-Net (src/AE.py:63-69) on what _find_side_information returned -> {"x_with_si": ...}."""
        x_dec, y_syn = found["x_dec"], found["y_syn"]
        if self.AE_only:
            return {"x_with_si": torch.zeros_like(y_syn)}
        y = y_syn
        fused = getattr(self._siNet, "fused", None)
        if fused is not None and hasattr(y_syn, "_dsin_nhwc"):
            x_with_si = fused(x_dec._dsin_nhwc, y_syn._dsin_nhwc, terms=self.precision.sinet)
        else:  # generic callable: normalise/concat/denormalise with torch elementwise ops
            mean, var = self.get_mean_var()
            m = torch.from_numpy(mean).to(y.device)
            s = torch.from_numpy(np.sqrt(var + 1e-10).astype(np.float32)).to(y.device)
            cat = torch.cat([(x_dec - m) / s, (y_syn - m) / s], dim=1)
            x_with_si = self._siNet(cat) * s + m
        return {"x_with_si": x_with_si}

    def _pinned_out(self, name, shape, dtype):
        key = ("out", name, self._ring, tuple(shape))
        buf = self._pinned.get(key)
        if buf is None:
            buf = torch.empty(tuple(shape), dtype=dtype, pin_memory=True)
            self._pinned[key] = buf
        return buf

    def siNet_get_reconstructed(self, x, y):
        """x, y: (B,3,H,W) arrays, uint8 (what the reference's DataProvider yields,
        src/DataProvider.py:197-199) or float32 holding uint8 values.  Returns numpy
        (y_dec, y_syn, x_dec, x_with_si, bpp) like src/AE.py:148.  The returned arrays are views of
        pinned staging buffers that are recycled two calls later.  The copy-out of y_dec/x_dec runs on
        a side stream while the SI-Finder is computing, that of y_syn while the SI-Net is.  With `use_cuda_graph` (default) the step is replayed from three CUDA graphs captured on the first call
        with this input shape (`use_cuda_graph = False` launches eagerly).  A batch of more than `e2e_chunk` pairs (a
        multiple of it) is processed as a software pipeline of chunks: host staging and H2D of chunk k+1 and the D2H of
        chunk k-1 overlap the kernels of chunk k (pairs are independent, so the results do not depend on the chunking)."""
        c = self.e2e_chunk
        if (self.use_cuda_graph and self.e2e_overlap and c and not torch.is_tensor(x) and not torch.is_tensor(y)
                and x.shape[0] > c and x.shape[0] % c == 0):
            return self._get_reconstructed_pipelined(np.ascontiguousarray(x), np.ascontiguousarray(y), int(c))
        xs, ys = self._stage(x, "x"), self._stage(y, "y")
        self._ring ^= 1
        main = torch.cuda.current_stream()
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        B = xs.shape[0]
        early = {}

        overlap = self.e2e_overlap

        def copy_out(name):
            """-> a hook that copies a finished segment's output to its pinned buffer on the side stream."""
            def hook(t):
                buf = self._pinned_out(name, t.shape, t.dtype)
                early[name] = buf
                if not overlap:
                    late.append((buf, t))
                    return
                self._copy_stream.wait_stream(main)
                with torch.cuda.stream(self._copy_stream):
                    buf.copy_(t, non_blocking=True)
                if not self.use_cuda_graph:  # graph outputs are static buffers; both streams are joined below
                    t.record_stream(self._copy_stream)
            return hook

        late = []
        on_decoded, on_found = copy_out("dec"), copy_out("y_syn")
        if self.use_cuda_graph:
            st = self._graph_state(B, xs.shape[2], xs.shape[3])
            st["x"].copy_(xs)  # uint8 -> fp32 conversion on the device, into the captured input buffers
            st["y"].copy_(ys)
            xd = st["x"]
            out = dict(st["out"])
            st["g_head"].replay()
            on_decoded(out["dec"])
            st["g_find"].replay()
            on_found(out["y_syn"])
            st["g_net"].replay()
        else:
            xd, yd = xs.to(torch.float32), ys.to(torch.float32)
            out = self.reconstruct_device(xd, yd, on_decoded=on_decoded, on_found=on_found)
        for buf, t in late:
            buf.copy_(t, non_blocking=True)
        last = self._pinned_out("x_with_si", out["x_with_si"].shape, out["x_with_si"].dtype)
        last.copy_(out["x_with_si"], non_blocking=True)
        bpp = bits.bitcost_to_bpp(out["bits"], xd)  # reads the fp64 bit sums (synchronises `main`)
        main.synchronize()
        self._copy_stream.synchronize()
        dec_host = early["dec"].numpy()
        self.last = out
        return dec_host[:B], early["y_syn"].numpy(), dec_host[B:], last.numpy(), bpp

    def _get_reconstructed_pipelined(self, x, y, c):
        """siNet_get_reconstructed for B = k * c pairs as a pipeline of k chunks of c pairs over three streams: `ins`
        (H2D of the next chunk), the current stream (the three captured graphs of a chunk + a device copy of each
        finished output into a private buffer), `cs` (D2H from the private buffers).  Events order the buffer reuse: an
        input slot is refilled only after the chunk that used it has converted it, a private output buffer is rewritten
        only after its previous D2H has finished.  Nothing blocks the host until the final synchronisation."""
        B, _, H, W = x.shape
        self._ring ^= 1
        main = torch.cuda.current_stream()
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        if self._in_stream is None:
            self._in_stream = torch.cuda.Stream()
        cs, ins = self._copy_stream, self._in_stream
        st = self._graph_state(c, H, W)
        out = st["out"]
        px = self._pinned_out("in_x", x.shape, torch.from_numpy(x[:0]).dtype)
        py = self._pinned_out("in_y", y.shape, torch.from_numpy(y[:0]).dtype)
        f32 = torch.float32
        host = {k: self._pinned_out(k, (B, 3, H, W), f32) for k in ("y_dec", "y_syn", "x_dec", "x_with_si")}
        key = (c, H, W, px.dtype, py.dtype)
        slots = self._dev_in.get(key)
        if slots is None:
            slots = [(torch.empty((c, 3, H, W), dtype=px.dtype, device=self.device),
                      torch.empty((c, 3, H, W), dtype=py.dtype, device=self.device)) for _ in range(2)]
            self._dev_in[key] = slots
        small = {k: torch.empty((B,) + tuple(out[k].shape[1:]), dtype=out[k].dtype, device=self.device)
                 for k in ("symbols", "symbols_y", "row", "col", "bits_sum", "best") if torch.is_tensor(out.get(k))}
        # D2H sources: private device buffers, two per output.  The graphs' own output tensors cannot be read by a copy
        # that overlaps the NEXT chunk: the three graphs share one memory pool, so e.g. x_with_si may occupy memory that
        # the first graph uses for an intermediate activation.
        okey = ("pipe_out", c, H, W)
        priv = self._dev_in.get(okey)
        if priv is None:
            priv = [{"dec": torch.empty_like(out["dec"]), "y_syn": torch.empty_like(out["y_syn"]),
                     "x_with_si": torch.empty_like(out["x_with_si"])} for _ in range(2)]
            self._dev_in[okey] = priv
        ins.wait_stream(main)  # the input slots may still be read by work the caller enqueued
        consumed = [None, None]   # per input slot: the chunk that used it has converted it
        drained = [{}, {}]        # per private output buffer: its D2H has finished
        for k in range(B // c):
            sl = slice(k * c, (k + 1) * c)
            _host_copy(px[sl], x[sl])
            _host_copy(py[sl], y[sl])
            dx, dy = slots[k % 2]
            if consumed[k % 2] is not None:
                ins.wait_event(consumed[k % 2])
            with torch.cuda.stream(ins):
                dx.copy_(px[sl], non_blocking=True)
                dy.copy_(py[sl], non_blocking=True)
                arrived = torch.cuda.Event()
                arrived.record(ins)
            main.wait_event(arrived)
            st["x"].copy_(dx)  # uint8 -> fp32 conversion on the device, into the captured input buffers
            st["y"].copy_(dy)
            consumed[k % 2] = torch.cuda.Event()
            consumed[k % 2].record(main)
            for seg, name in (("g_head", "dec"), ("g_find", "y_syn"), ("g_net", "x_with_si")):
                st[seg].replay()
                if seg == "g_head":
                    for kk, t in small.items():
                        if kk in ("symbols", "symbols_y", "bits_sum"):
                            t[sl].copy_(out[kk])
                elif seg == "g_find":
                    for kk, t in small.items():
                        if kk in ("row", "col", "best"):
                            t[sl].copy_(out[kk])
                src = priv[k % 2][name]
                if name in drained[k % 2]:
                    main.wait_event(drained[k % 2][name])  # chunk k-2's D2H of this buffer (long finished)
                src.copy_(out[name])
                ready = torch.cuda.Event()
                ready.record(main)
                cs.wait_event(ready)
                with torch.cuda.stream(cs):
                    if name == "dec":
                        host["y_dec"][sl].copy_(src[:c], non_blocking=True)
                        host["x_dec"][sl].copy_(src[c:], non_blocking=True)
                    else:
                        host[name][sl].copy_(src, non_blocking=True)
                    drained[k % 2][name] = torch.cuda.Event()
                    drained[k % 2][name].record(cs)
        main.synchronize()
        cs.synchronize()
        num_bits = float(small["bits_sum"].sum().item())
        bpp = np.float32(num_bits / float(B * H * W))  # bits.bitcost_to_bpp over the whole batch
        self.last = small
        return host["y_dec"].numpy(), host["y_syn"].numpy(), host["x_dec"].numpy(), host["x_with_si"].numpy(), bpp

    # ------------------------------------------------------------------ real bitstreams (SURVEY 8f N3)
    def compress(self, x, nstreams=8):
        """x (B,3,H,W) uint8 / uint8-valued array -> list of B bitstreams (bytes).  Encoder + quantiser
        (src/AE.py:50-53) followed by the PC1 range coder driven by the probability model
        (the coder src/probclass_imgcomp.py:361-482 prepares for); 8 * len(bitstream) / (H * W) is the real bpp
        that `bpp` of siNet_get_reconstructed estimates."""
        xd = self._to_device(x, "x")
        z = self._encode(xd, self.ae_imgcomp, is_training=False, terms=self.precision.enc_x)
        self.last = {"symbols": z.symbols, "qbar": z.qbar}
        return self.pc_imgcomp.encode_symbols(z.symbols, self.ae_imgcomp._centers, nstreams=nstreams)

    def decompress(self, bitstreams, y):
        """Receiver: bitstreams of B images + the side images y (B,3,H,W) -> numpy (y_dec, y_syn, x_dec, x_with_si),
        i.e. src/AE.py:132-148 without access to x.  The decoder input is qhard = centres[symbols]; the sender-side
        graph feeds qbar = qsoft + (qhard - qsoft), which equals qhard up to one fp32 rounding."""
        yd = self._to_device(y, "y")
        f = self.ae_imgcomp.get_subsampling_factor()
        sym = self.pc_imgcomp.decode_symbols(list(bitstreams), self.ae_imgcomp._centers, expect_shape=(
            self.ae_config.num_chan_bn, yd.shape[2] // f, yd.shape[3] // f))
        if sym.shape[0] != yd.shape[0]:
            raise ValueError("{} bitstreams for {} side images".format(sym.shape[0], yd.shape[0]))
        qhard = self.ae_imgcomp._centers[sym]
        out = self.decode_side_device(qhard.contiguous(), yd)
        out["symbols"] = sym
        self.last = out
        return tuple(self._to_host([out[k] for k in ("y_dec", "y_syn", "x_dec", "x_with_si")]))

    def create_y_dec(self, y):
        yd = self._to_device(y, "y")
        z = self._encode(yd, self.ae_imgcomp, is_training=False, terms=self.precision.enc_y)
        dec = self._decode(z.qbar, self.ae_imgcomp, is_training=False, terms=self.precision.dec)
        return self._to_host([dec])[0]
