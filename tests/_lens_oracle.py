"""CPU restatement of latent-bokeh's lens-conditioned ConditionalNAFNet (tests/ is on sys.path under pytest's default
import mode).  TEST INFRASTRUCTURE ONLY, like oracle/irsde_oracle.py, whose layer helpers it reuses; pinned to the
reference by tests/golden/reference_golden_lens.pt (tests/test_lens_host.py).  File:line citations are relative to
codes/config/latent-bokeh/models/modules/DenoisingNAFNet_arch.py of the reference checkout."""
import math

import torch
import torch.nn.functional as F

from oracle import irsde_oracle as O


def nafnet_lens_param_shapes(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums):
    """State-dict names -> shapes in the reference's registration order (:15-53,95-155): the plain NAFNet's, with
    time_mlp.0/.2 at the top (the embedding is applied outside the Sequential, :102-107), cam_mlp.0/.2 after it (:109-113),
    and in every block time_mlp.1 (was mlp.1) followed by cam_mlp.1 (:18-24)."""
    td = width * 4
    S = {}
    for name, shp in O.nafnet_param_shapes(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums).items():
        if name == "time_mlp.1.weight":
            S["time_mlp.0.weight"] = shp
        elif name == "time_mlp.1.bias":
            S["time_mlp.0.bias"] = shp
        elif name == "time_mlp.3.weight":
            S["time_mlp.2.weight"] = shp
        elif name == "time_mlp.3.bias":
            S["time_mlp.2.bias"] = shp
            S["cam_mlp.0.weight"] = (td * 2, width * 3)
            S["cam_mlp.0.bias"] = (td * 2,)
            S["cam_mlp.2.weight"] = (td, td)
            S["cam_mlp.2.bias"] = (td,)
        elif name.endswith("mlp.1.weight"):
            S[name.replace("mlp.1.", "time_mlp.1.")] = shp
        elif name.endswith("mlp.1.bias"):
            pre = name[:-len("mlp.1.bias")]
            S[pre + "time_mlp.1.bias"] = shp
            c = shp[0] // 4
            S[pre + "cam_mlp.1.weight"] = (2 * c, td // 2)
            S[pre + "cam_mlp.1.bias"] = (2 * c,)
        else:
            S[name] = shp
    return S


def make_nafnet_lens_weights(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums, seed=0):
    """Seeded random weights, same recipe as O.make_nafnet_weights."""
    g = torch.Generator().manual_seed(seed)
    P = {}
    for name, shp in nafnet_lens_param_shapes(img_channel, width, middle_blk_num, enc_blk_nums, dec_blk_nums).items():
        if name.endswith(".g"):
            P[name] = 1.0 + 0.1 * torch.randn(shp, generator=g)
        elif name.endswith("beta") or name.endswith("gamma"):
            P[name] = 0.5 * torch.randn(shp, generator=g)  # reference inits these to zero (identity blocks)
        elif name.endswith("bias"):
            P[name] = 0.05 * torch.randn(shp, generator=g)
        else:
            fan_in = 1
            for d in shp[1:]:
                fan_in *= d
            P[name] = (torch.rand(shp, generator=g) * 2 - 1) * math.sqrt(3.0 / fan_in)
    return P


def _sinus(v, width):
    """SinusoidalPosEmb(width) (module_util.py:36-48)."""
    half = width // 2
    freqs = torch.exp(torch.arange(half) * -(math.log(10000) / (half - 1)))
    e = v[:, None] * freqs[None, :]
    return torch.cat((e.sin(), e.cos()), dim=-1)


def naf_lens_block(P, pre, x, t, cam):
    """NAFBlock.forward (:60-90): time chunks (shift_att, scale_att, shift_ffn, scale_ffn), camera chunks (scale, shift),
    x * (cam_scale + 1) + cam_shift right after the FFN SimpleGate (:82-83)."""
    te = F.linear(O._gate(t, dim=-1), P[pre + "time_mlp.1.weight"], P[pre + "time_mlp.1.bias"])[:, :, None, None]
    shift_att, scale_att, shift_ffn, scale_ffn = te.chunk(4, dim=1)
    ce = F.linear(O._gate(cam, dim=-1), P[pre + "cam_mlp.1.weight"], P[pre + "cam_mlp.1.bias"])[:, :, None, None]
    cam_scale, cam_shift = ce.chunk(2, dim=1)
    inp = x
    x = O.layer_norm_c(x, P[pre + "norm1.g"])
    x = x * (scale_att + 1) + shift_att
    x = F.conv2d(x, P[pre + "conv1.weight"], P[pre + "conv1.bias"])
    x = F.conv2d(x, P[pre + "conv2.weight"], P[pre + "conv2.bias"], padding=1, groups=x.shape[1])
    x = O._gate(x)
    pooled = x.mean(dim=(2, 3), keepdim=True)
    x = x * F.conv2d(pooled, P[pre + "sca.1.weight"], P[pre + "sca.1.bias"])
    x = F.conv2d(x, P[pre + "conv3.weight"], P[pre + "conv3.bias"])
    y = inp + x * P[pre + "beta"]
    x = O.layer_norm_c(y, P[pre + "norm2.g"])
    x = x * (scale_ffn + 1) + shift_ffn
    x = F.conv2d(x, P[pre + "conv4.weight"], P[pre + "conv4.bias"])
    x = O._gate(x)
    x = x * (cam_scale + 1) + cam_shift
    x = F.conv2d(x, P[pre + "conv5.weight"], P[pre + "conv5.bias"])
    return y + x * P[pre + "gamma"]


def nafnet_lens_forward(P, inp, cond, time, lens, width, enc_blk_nums, middle_blk_num, dec_blk_nums):
    """ConditionalNAFNet.forward (:159-199).  ``lens`` = [src_lens, tgt_lens, disparity]: numbers, 1-element or [B]
    tensors (1-element entries shared by the batch); cam_embed = cam_mlp(cat(SinusoidalPosEmb(w)(entry))) (:171-173);
    plain ending(x) (:195)."""
    if isinstance(time, (int, float)):
        time = torch.tensor([time])
    time = time.reshape(-1)
    x = torch.cat([inp - cond, cond], dim=1)
    t = F.linear(_sinus(time, width), P["time_mlp.0.weight"], P["time_mlp.0.bias"])
    t = F.linear(O._gate(t, dim=-1), P["time_mlp.2.weight"], P["time_mlp.2.bias"])
    cols = [torch.as_tensor(v).reshape(-1) for v in lens]
    n = max(c.numel() for c in cols)
    cam = torch.cat([_sinus(c.expand(n), width) for c in cols], dim=1)
    cam = F.linear(cam, P["cam_mlp.0.weight"], P["cam_mlp.0.bias"])
    cam = F.linear(O._gate(cam, dim=-1), P["cam_mlp.2.weight"], P["cam_mlp.2.bias"])
    H, W = x.shape[2:]
    s = 2 ** len(enc_blk_nums)
    x = F.pad(x, (0, (s - W % s) % s, 0, (s - H % s) % s))  # zero pad (check_image_size, :201-206)
    x = F.conv2d(x, P["intro.weight"], P["intro.bias"], padding=1)
    encs = []
    for i, num in enumerate(enc_blk_nums):
        for j in range(num):
            x = naf_lens_block(P, "encoders.%d.%d." % (i, j), x, t, cam)
        encs.append(x)
        x = F.conv2d(x, P["downs.%d.weight" % i], P["downs.%d.bias" % i], stride=2)
    for j in range(middle_blk_num):
        x = naf_lens_block(P, "middle_blks.%d." % j, x, t, cam)
    for i, num in enumerate(dec_blk_nums):
        x = F.pixel_shuffle(F.conv2d(x, P["ups.%d.0.weight" % i]), 2)
        x = x + encs[len(encs) - 1 - i]
        for j in range(num):
            x = naf_lens_block(P, "decoders.%d.%d." % (i, j), x, t, cam)
    x = F.conv2d(x, P["ending.weight"], P["ending.bias"], padding=1)
    return x[..., :H, :W]
