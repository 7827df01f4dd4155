"""Golden fixture for the lens-conditioned ConditionalNAFNet of latent-bokeh (Refusion's bokeh score network,
codes/config/latent-bokeh/models/modules/DenoisingNAFNet_arch.py), generated from the imported reference on the CPU.
    python tests/golden/make_golden_lens.py
"""
import importlib.util
import os
import sys

import torch

REF = "/root/reference/codes"
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, OUT)
from make_golden_nafnet import load_arch  # noqa: E402


def load_sde_utils():
    """codes/utils/sde_utils.py by file path (the `utils` package __init__ pulls in image / file helpers not needed here)."""
    spec = importlib.util.spec_from_file_location("ref_sde_utils", os.path.join(REF, "utils", "sde_utils.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def main():
    torch.set_num_threads(4)
    g = torch.Generator().manual_seed(21)
    arch = load_arch("latent-bokeh")
    cfg = dict(img_channel=4, width=8, middle_blk_num=1, enc_blk_nums=[1, 2], dec_blk_nums=[1, 1])
    torch.manual_seed(4)
    net = arch.ConditionalNAFNet(**cfg).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    for k in sd:  # beta/gamma are zero-initialised in the reference: make every branch matter
        if k.endswith("beta") or k.endswith("gamma"):
            sd[k] = 0.5 * torch.randn(sd[k].shape, generator=g)
        if k.endswith(".g"):
            sd[k] = 1 + 0.2 * torch.randn(sd[k].shape, generator=g)
    net.load_state_dict(sd)
    x = torch.rand(2, 4, 18, 23, generator=g)
    cond = torch.rand(2, 4, 18, 23, generator=g)
    # BokehLQGT_dataset.py:101-105: lens strings -> f-number * 10 (Canon50mmf1.8 -> -18, Sony50mmf16 -> 160), disparity as
    # read; the DataLoader hands each over as a 1-element tensor at batch 1
    lens_int = [torch.tensor([-18.0]), torch.tensor([160.0]), torch.tensor([3.5])]
    lens_vec = [torch.tensor([-18.0, 160.0]), torch.tensor([160.0, 18.0]), torch.tensor([3.5, 12.0])]
    t_vec = torch.tensor([3, 40])
    with torch.no_grad():
        y_int = net(x[:1], cond[:1], 13, lens_info=lens_int)
        y_vec = net(x, cond, t_vec, lens_info=lens_vec)

    # the reference's own sampler: IRSDE.reverse_sde(..., lens_info=...) (sde_utils.py:252-266), every torch.randn_like draw
    # of the T steps (dispersion, sde_utils.py:39-41) served from the stored table z in loop order
    sde_utils = load_sde_utils()
    T, max_sigma, eps = 8, 50, 0.005
    sde = sde_utils.IRSDE(max_sigma=max_sigma, T=T, schedule="cosine", eps=eps, device="cpu")
    sde.set_model(net)
    lq = torch.rand(1, 4, 18, 23, generator=g)
    sde.set_mu(lq)
    xT = lq + torch.randn(lq.shape, generator=g) * sde.max_sigma
    zs = torch.randn((T,) + tuple(lq.shape), generator=g)
    draws = iter(zs)
    randn_like = torch.randn_like
    torch.randn_like = lambda a, *args, **kw: next(draws).clone()
    try:
        with torch.no_grad():
            x0 = sde.reverse_sde(xT, lens_info=lens_int)
    finally:
        torch.randn_like = randn_like
    assert next(draws, None) is None, "the chain must consume exactly T draws"

    gold = dict(cfg=cfg, state=sd, x=x, cond=cond, t_int=13, lens_int=lens_int, y_int=y_int, t_vec=t_vec, lens_vec=lens_vec,
                y_vec=y_vec, chain=dict(T=T, max_sigma=max_sigma, eps=eps, lq=lq, xT=xT, zs=zs, lens=lens_int, x0=x0))
    path = os.path.join(OUT, "reference_golden_lens.pt")
    torch.save(gold, path)
    print("wrote", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
