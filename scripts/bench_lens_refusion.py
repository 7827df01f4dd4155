"""Refusion latent-bokeh (codes/config/latent-bokeh/options/bokeh/test/refusion.yml) on one GPU, seeded random weights:
latent UNet(3, 3, ch 64, ch_mult [1, 2, 4], embed_dim 4) encode -> lens-conditioned ConditionalNAFNet(img_channel 4, width 64,
enc [2, 2, 4, 8], mid 12, dec [2, 2, 2, 2]) reverse_sde(T = 100, lens_info=...) -> decode, on one 1x3x1440x1920 image.

Prints one JSON line: chain ms and img/s, end-to-end img/s (encode + chain + decode), launches per sampler step, the card
and its power limit, and the cost of the camera conditioning: chains of the lens network and of the same-shaped
unconditioned ConditionalNAFNet(img_channel=4) alternated A, B, A, B in this one process (CUDA-event times, medians).
Needs a CUDA device; there is no CPU fallback.

    python scripts/bench_lens_refusion.py [--T 100] [--height 1440] [--width 1920] [--rounds 3] [--precision bf16]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NAF = dict(img_channel=4, width=64, enc_blk_nums=[2, 2, 4, 8], middle_blk_num=12, dec_blk_nums=[2, 2, 2, 2])
AE = dict(in_ch=3, out_ch=3, ch=64, ch_mult=[1, 2, 4], embed_dim=4)
LENS = [-18.0, 160.0, 3.5]  # (src_lens, tgt_lens, disparity) as BokehLQ_dataset yields them: f-number * 10, disparity


def latent_hw(H, W):
    """Latent size of UNet.encode (UNet_arch.py:59-76): pad to 2^len(ch_mult), then len(ch_mult) - 1 stride-2 stages."""
    d = len(AE["ch_mult"])
    s = 1 << d
    return (H + (s - H % s) % s) >> (d - 1), (W + (s - W % s) % s) >> (d - 1)


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--height", type=int, default=1440)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--rounds", type=int, default=3, help="alternated (lens, plain) chain pairs")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "fp32x3"])
    args = ap.parse_args()
    if args.T < 1 or args.rounds < 1:
        raise SystemExit("--T and --rounds must be >= 1")
    lat_h, lat_w = latent_hw(args.height, args.width)
    image = [1, 3, args.height, args.width]
    latent = [1, NAF["img_channel"], lat_h, lat_w]

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_lens_refusion: no GPU - this benchmark runs the CUDA library on a B200 and has no CPU path "
                         "(image %s, latent %s)" % (image, latent))
    import irsde_b200

    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(0)
    torch.manual_seed(0)
    ae = irsde_b200.UNet(precision=args.precision, **AE).to(dev)
    nets = {}
    for name, lens in (("lens", True), ("plain", False)):
        torch.manual_seed(1)
        net = irsde_b200.ConditionalNAFNet(lens=lens, precision=args.precision, **NAF)
        with torch.no_grad():
            for pname, p in net.named_parameters():
                if pname.endswith("beta") or pname.endswith("gamma"):  # zero-initialised (identity blocks) in the reference
                    p.copy_(0.1 * torch.randn(p.shape, generator=g))
        nets[name] = net.to(dev)
    sdes = {}
    for name, net in nets.items():
        sde = irsde_b200.IRSDE(max_sigma=50, T=args.T, schedule="cosine", eps=0.005, device=dev)
        sde.set_model(net)
        sde.rng = "philox"  # in-kernel noise: no per-step randn_like in the timed window
        sdes[name] = sde
    x = torch.rand(*image, generator=g).to(dev)
    lens_info = [torch.tensor([v]) for v in LENS]

    def chain(name, xT):
        return sdes[name].reverse_sde(xT, lens_info=lens_info) if name == "lens" else sdes[name].reverse_sde(xT)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    z, h = ae.encode(x)
    assert list(z.shape) == latent, (list(z.shape), latent)
    for sde in sdes.values():
        sde.set_mu(z)
    xT = sdes["lens"].noise_state(z)
    launches = {}
    for name in ("lens", "plain"):  # warm-up: plan build, step-graph capture, camera rows
        l0 = nets[name].launch_count()
        chain(name, xT)
        torch.cuda.synchronize()
        l1 = nets[name].launch_count()
        chain(name, xT)
        torch.cuda.synchronize()
        launches[name] = (nets[name].launch_count() - l1) / args.T  # a steady chain, incl. its 3 per-chain launches
    runs = {"lens": [], "plain": []}
    for _ in range(args.rounds):
        for name in ("lens", "plain"):
            ms, z0 = timed(lambda: chain(name, xT))
            runs[name].append(ms)
            assert torch.isfinite(z0).all(), name

    def e2e():
        zz, hh = ae.encode(x)
        sdes["lens"].set_mu(zz)
        return ae.decode(chain("lens", sdes["lens"].noise_state(zz)), hh)

    e2e()
    e2e_ms = []
    for _ in range(args.rounds):
        ms, y = timed(e2e)
        e2e_ms.append(ms)
    assert torch.isfinite(y).all() and list(y.shape) == image

    lens_ms, plain_ms = statistics.median(runs["lens"]), statistics.median(runs["plain"])
    e2e_med = statistics.median(e2e_ms)
    print(json.dumps({
        "workload": "latent-bokeh refusion: UNet encode -> lens ConditionalNAFNet reverse_sde -> decode",
        "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "precision": args.precision,
        "image": image, "latent": latent, "T": args.T, "rounds": args.rounds,
        "chain_ms": round(lens_ms, 2), "chain_img_per_s": round(1e3 / lens_ms, 4), "ms_per_step": round(lens_ms / args.T, 4),
        "e2e_ms": round(e2e_med, 2), "e2e_img_per_s": round(1e3 / e2e_med, 4),
        "launches_per_step": round(launches["lens"], 2), "plain_launches_per_step": round(launches["plain"], 2),
        "plain_chain_ms": round(plain_ms, 2),
        "conditioning_cost_pct": round(100.0 * (lens_ms - plain_ms) / plain_ms, 2),
        "chain_ms_runs": {k: [round(v, 2) for v in vs] for k, vs in runs.items()},
        "e2e_ms_runs": [round(v, 2) for v in e2e_ms],
    }))


if __name__ == "__main__":
    main()
