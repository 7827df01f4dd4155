"""``ConditionalNAFNet`` (Refusion's score network) with the reference's constructor, ``forward(inp, cond, time)``
signature and state-dict names/shapes (codes/config/deraining/models/modules/DenoisingNAFNet_arch.py:87-188; latent
variant codes/config/latent-dehazing/models/modules/DenoisingNAFNet_arch.py:147-181; lens-conditioned variant
codes/config/latent-bokeh/models/modules/DenoisingNAFNet_arch.py:93-199, ``forward(inp, cond, time, lens_info=...)``),
executed by the native library.
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib
from .unet import ConditionalUNet, _Node


def nafnet_param_shapes(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums, lens=False):
    """State-dict entries in the reference's registration order (DenoisingNAFNet_arch.py:15-49,89-143).  ``lens``: the
    latent-bokeh variant (latent-bokeh/.../DenoisingNAFNet_arch.py:18-24,102-113): ``time_mlp.0/.2`` and ``cam_mlp.0/.2`` at
    the top, ``time_mlp.1`` and ``cam_mlp.1`` in every block."""
    S = {}
    td = width * 4
    t1, t3 = ("time_mlp.0.", "time_mlp.2.") if lens else ("time_mlp.1.", "time_mlp.3.")
    S[t1 + "weight"] = (td * 2, width)
    S[t1 + "bias"] = (td * 2,)
    S[t3 + "weight"] = (td, td)
    S[t3 + "bias"] = (td,)
    if lens:
        S["cam_mlp.0.weight"] = (td * 2, width * 3)
        S["cam_mlp.0.bias"] = (td * 2,)
        S["cam_mlp.2.weight"] = (td, td)
        S["cam_mlp.2.bias"] = (td,)
    S["intro.weight"] = (width, img_channel * 2, 3, 3)
    S["intro.bias"] = (width,)
    S["ending.weight"] = (img_channel, width, 3, 3)
    S["ending.bias"] = (img_channel,)

    def blk(pre, c):
        S[pre + "beta"] = (1, c, 1, 1)
        S[pre + "gamma"] = (1, c, 1, 1)
        mlp = pre + ("time_mlp.1." if lens else "mlp.1.")
        S[mlp + "weight"] = (4 * c, td // 2)
        S[mlp + "bias"] = (4 * c,)
        if lens:
            S[pre + "cam_mlp.1.weight"] = (2 * c, td // 2)
            S[pre + "cam_mlp.1.bias"] = (2 * c,)
        for name, shp in (("conv1", (2 * c, c, 1, 1)), ("conv2", (2 * c, 1, 3, 3)), ("conv3", (c, c, 1, 1)),
                          ("sca.1", (c, c, 1, 1)), ("conv4", (2 * c, c, 1, 1)), ("conv5", (c, c, 1, 1))):
            S[pre + name + ".weight"] = shp
            S[pre + name + ".bias"] = (shp[0],)
        S[pre + "norm1.g"] = (1, c, 1, 1)
        S[pre + "norm2.g"] = (1, c, 1, 1)

    chan = width
    for i, num in enumerate(enc_blk_nums):
        for j in range(num):
            blk("encoders.%d.%d." % (i, j), chan)
        chan *= 2
    mid_c = chan
    for i, num in enumerate(dec_blk_nums):
        chan //= 2
        for j in range(num):
            blk("decoders.%d.%d." % (i, j), chan)
    for j in range(middle_blk_num):
        blk("middle_blks.%d." % j, mid_c)
    chan = mid_c
    for i in range(len(dec_blk_nums)):
        S["ups.%d.0.weight" % i] = (chan * 2, chan, 1, 1)
        chan //= 2
    chan = width
    for i in range(len(enc_blk_nums)):
        S["downs.%d.weight" % i] = (chan * 2, chan, 2, 2)
        S["downs.%d.bias" % i] = (chan * 2,)
        chan *= 2
    return S


class _NafConfig(ctypes.Structure):
    _fields_ = [("img_channel", ctypes.c_int32), ("width", ctypes.c_int32), ("middle_blk_num", ctypes.c_int32),
                ("n_levels", ctypes.c_int32), ("enc_blk_nums", ctypes.c_int32 * 8), ("dec_blk_nums", ctypes.c_int32 * 8),
                ("latent", ctypes.c_int32), ("precision", ctypes.c_int32), ("device", ctypes.c_int32),
                ("flags", ctypes.c_int32)]


class _NafContext(_lib.Context):
    def __init__(self, img_channel, width, middle, enc, dec, latent, precision, device_index, force_simt=False, lens=False):
        L = _lib.load()
        create = L.irsde_create_nafnet_lens if lens else L.irsde_create_nafnet
        create.argtypes = [ctypes.POINTER(_NafConfig), ctypes.POINTER(ctypes.c_void_p)]
        create.restype = ctypes.c_int
        cfg = _NafConfig(img_channel, width, middle, len(enc), (ctypes.c_int32 * 8)(*enc), (ctypes.c_int32 * 8)(*dec),
                         1 if latent else 0, precision, device_index, 1 if force_simt else 0)
        h = ctypes.c_void_p()
        _lib.check(create(ctypes.byref(cfg), ctypes.byref(h)))
        self.h = h
        self.L = L


class ConditionalNAFNet(ConditionalUNet):
    """Drop-in for the reference ``ConditionalNAFNet``.  ``latent=True`` selects the latent-dehazing variant
    (``ending(x + intro(x))``); ``lens=True`` the latent-bokeh variant, whose blocks are also modulated by a camera
    embedding of ``lens_info = [src_lens, tgt_lens, disparity]`` (``forward(inp, cond, time, lens_info=...)``).
    Inherits weight upload / forward plumbing from ``ConditionalUNet``."""

    variant = "conditional"

    def __init__(self, img_channel=3, width=16, middle_blk_num=1, enc_blk_nums=[], dec_blk_nums=[], upscale=1,
                 latent=False, precision=None, force_simt=False, lens=False):
        nn.Module.__init__(self)
        import os
        if len(enc_blk_nums) != len(dec_blk_nums) or len(enc_blk_nums) > 8:
            raise ValueError("enc_blk_nums / dec_blk_nums must have the same length (<= 8)")
        if lens and latent:
            raise ValueError("the lens network ends in a plain ending(x): latent must be False")
        self.lens = bool(lens)
        self.in_nc = self.out_nc = img_channel
        self.img_channel, self.width, self.middle_blk_num = img_channel, width, middle_blk_num
        self.enc_blk_nums, self.dec_blk_nums = list(enc_blk_nums), list(dec_blk_nums)
        self.upscale, self.latent = upscale, latent
        self.precision = precision or os.environ.get("IRSDE_B200_PRECISION", "fp32")
        if self.precision not in _lib.PRECISIONS:
            raise ValueError("precision must be one of %s" % (sorted(_lib.PRECISIONS),))
        self._force_simt = force_simt
        self._shapes = nafnet_param_shapes(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums, self.lens)
        for name, shp in self._shapes.items():
            parts = name.split(".")
            node = self
            for p in parts[:-1]:
                if p not in node._modules:
                    node.add_module(p, _Node())
                node = node._modules[p]
            if name.endswith("beta") or name.endswith("gamma"):
                init = torch.zeros(shp)  # reference: zeros (DenoisingNAFNet_arch.py:45-46)
            else:
                init = self._init(name, shp)
            node.register_parameter(parts[-1], nn.Parameter(init))
        self._ctx = None
        self._ctx_dev = None
        self._sig = None

    def _context(self, device):
        if device.type != "cuda":
            raise RuntimeError("irsde_b200.ConditionalNAFNet runs on CUDA (sm_100a) only; there is no CPU path")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self._ctx is None or self._ctx_dev != idx:
            if self._ctx is not None:
                self._ctx.close()
            self._ctx = _NafContext(self.img_channel, self.width, self.middle_blk_num, self.enc_blk_nums, self.dec_blk_nums,
                                    self.latent, _lib.PRECISIONS[self.precision], idx,
                                    force_simt=self._force_simt, lens=self.lens)
            self._ctx_dev = idx
            self._sig = None
        return self._ctx

    @staticmethod
    def lens_rows(lens_info):
        """``[src_lens, tgt_lens, disparity]`` -> host float32 ``[n][3]``.  Each entry is a Python number, a 1-element tensor
        (what the DataLoader yields at batch 1) or an ``[n]`` tensor, on any device; 1-element entries are shared by the
        batch."""
        if len(lens_info) != 3:
            raise ValueError("lens_info must hold 3 entries [src_lens, tgt_lens, disparity], got %d" % len(lens_info))
        cols = [torch.as_tensor(v).detach().reshape(-1).float().cpu() for v in lens_info]
        n = max(c.numel() for c in cols)
        if any(c.numel() not in (1, n) for c in cols):
            raise ValueError("lens_info entries must hold 1 or the same number of values")
        return torch.stack([c.expand(n) for c in cols], dim=1).contiguous()

    def set_lens(self, lens_info, device):
        """Camera rows of the following forwards / chains on ``device`` (irsde_set_lens): one row shared by the batch, or one
        per image, where image b's result is the network run on image b alone with its own lens."""
        self._upload_lens(self.lens_rows(lens_info), device)

    def _upload_lens(self, rows, device):
        ctx = self.sync_weights(device)
        arr = _lib.float_array(rows.reshape(-1).tolist())
        with torch.cuda.device(device):
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(ctx.L.irsde_set_lens(ctx.h, arr, rows.shape[0], ctypes.c_void_p(st)), ctx.h)

    @torch.no_grad()
    def forward(self, inp, cond, time, **kwargs):
        if not self.lens:
            if kwargs:
                raise TypeError("forward() got an unexpected keyword argument %r" % next(iter(kwargs)))
            return self._run(inp, cond, time)
        rows = self.lens_rows(kwargs["lens_info"])  # KeyError('lens_info') without it, as the reference (:161)
        if not inp.is_cuda:
            raise RuntimeError("irsde_b200.ConditionalNAFNet runs on CUDA (sm_100a) only; there is no CPU path")
        self._upload_lens(rows, inp.device)
        return self._run(inp, cond, time)
