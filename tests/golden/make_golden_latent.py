"""Golden fixture for the Refusion latent autoencoder UNet.encode/decode, generated from the imported reference
(random small configuration).    python tests/golden/make_golden_latent.py"""
import importlib.util
import os
import sys
import types

import torch

REF = "/root/reference/codes"
OUT = os.path.dirname(os.path.abspath(__file__))


def load_unet_arch():
    base = os.path.join(REF, "config", "latent-dehazing", "models", "modules")
    pkg = types.ModuleType("refmods_latent")
    pkg.__path__ = [base]
    sys.modules[pkg.__name__] = pkg
    out = {}
    for name in ("module_util", "UNet_arch"):
        spec = importlib.util.spec_from_file_location(pkg.__name__ + "." + name, os.path.join(base, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = m
        spec.loader.exec_module(m)
        out[name] = m
    return out["UNet_arch"]


def main():
    arch = load_unet_arch()
    g = torch.Generator().manual_seed(9)
    cfg = dict(in_ch=3, out_ch=3, ch=8, ch_mult=[2, 4], embed_dim=4)
    torch.manual_seed(4)
    net = arch.UNet(**cfg).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    for k in sd:
        if k.endswith(".g"):
            sd[k] = 1 + 0.2 * torch.randn(sd[k].shape, generator=g)
        if k.endswith("bias"):
            sd[k] = sd[k] + 0.05 * torch.randn(sd[k].shape, generator=g)
    net.load_state_dict(sd)
    x = torch.rand(2, 3, 21, 30, generator=g)
    with torch.no_grad():
        z, h = net.encode(x)
        z2 = z + 0.1 * torch.randn(z.shape, generator=g)   # what the latent sampler would hand back
        y = net.decode(z2, h)
        y_id = net.decode(z, h)
    gold = dict(cfg=cfg, state=sd, x=x, z=z, z2=z2, y=y, y_id=y_id)
    torch.save(gold, os.path.join(OUT, "reference_golden_latent.pt"))
    print("wrote", os.path.getsize(os.path.join(OUT, "reference_golden_latent.pt")))


if __name__ == "__main__":
    main()
