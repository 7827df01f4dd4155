"""GPU tests (B200) of the lens-conditioned ConditionalNAFNet (latent-bokeh): forwards and the reference's own sampler
chain against tests/golden/reference_golden_lens.pt, bf16 against the oracle, graph replay against eager launches, batch
independence of per-image lens, re-use of one plan across lens changes, and the error contract of the C ABI."""
import ctypes
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import _lens_oracle as L  # noqa: E402


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _maxdiff(a, b):
    return (a.detach().float().cpu() - b.detach().float().cpu()).abs().max().item()


@pytest.fixture(scope="module")
def lib():
    import irsde_b200
    return irsde_b200


@pytest.fixture(scope="module")
def gl():
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_golden_lens.pt"), weights_only=True)


def _net(lib, gl, precision):
    net = lib.ConditionalNAFNet(lens=True, precision=precision, **gl["cfg"])
    net.load_state_dict(gl["state"], strict=True)
    return net.to(_dev())


def _sde(lib, gl, net, lq):
    ch = gl["chain"]
    sde = lib.IRSDE(ch["max_sigma"], ch["T"], schedule="cosine", eps=ch["eps"], device=_dev())
    sde.set_model(net)
    sde.set_mu(lq.to(_dev()))
    return sde


def _args(c):
    return c["width"], c["enc_blk_nums"], c["middle_blk_num"], c["dec_blk_nums"]


@pytest.mark.parametrize("precision", ["fp32", "fp32x3"])
def test_lens_forward_vs_reference(lib, gl, precision):
    """fp32 and fp32x3 vs the reference's own outputs (< 1e-4): B = 1 with int t and 1-element lens tensors, B = 2 with
    per-image t and per-image lens (zero pad 18x23 -> 20x24)."""
    dev = _dev()
    net = _net(lib, gl, precision)
    y = net(gl["x"][:1].to(dev), gl["cond"][:1].to(dev), gl["t_int"], lens_info=gl["lens_int"])
    assert _maxdiff(y, gl["y_int"]) < 1e-4
    lens_dev = [v.to(dev) for v in gl["lens_vec"]]  # lens tensors on the GPU are accepted as well
    yv = net(gl["x"].to(dev), gl["cond"].to(dev), gl["t_vec"], lens_info=lens_dev)
    assert _maxdiff(yv, gl["y_vec"]) < 1e-4


def test_lens_forward_bf16_vs_oracle(lib, gl):
    """bf16 perf mode vs the oracle: <= 4 % of the output scale, shared and per-image lens."""
    dev = _dev()
    net = _net(lib, gl, "bf16")
    for lens, t in ((gl["lens_int"], 13), (gl["lens_vec"], gl["t_vec"])):
        yo = L.nafnet_lens_forward(gl["state"], gl["x"], gl["cond"], t, lens, *_args(gl["cfg"]))
        yb = net(gl["x"].to(dev), gl["cond"].to(dev), t, lens_info=lens)
        assert _maxdiff(yb, yo) <= 4e-2 * yo.abs().max().item()


def test_lens_chain_vs_reference_and_eager(lib, gl):
    """fp32 reverse_sde(..., lens_info=...) through the captured step graph vs the reference's own chain (< 1e-3), and the
    graph replay equals eager per-step launches (use_graph=False) bit for bit."""
    dev = _dev()
    ch = gl["chain"]
    net = _net(lib, gl, "fp32")
    sde = _sde(lib, gl, net, ch["lq"])
    assert sde._fast({"lens_info": ch["lens"]}, False)
    x0 = sde.reverse_sde(ch["xT"].to(dev), zs=ch["zs"].to(dev), lens_info=ch["lens"])
    assert _maxdiff(x0, ch["x0"]) < 1e-3
    sde.use_graph = False
    x0e = sde.reverse_sde(ch["xT"].to(dev), zs=ch["zs"].to(dev), lens_info=ch["lens"])
    assert torch.equal(x0.cpu(), x0e.cpu())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_lens_batch_independence(lib, gl, precision):
    """B = 2 with different per-image lens (and t) equals two B = 1 runs bit for bit: the forward, and a Philox chain (noise
    keyed by image uid, so image 1 alone runs with image base 1)."""
    dev = _dev()
    net = _net(lib, gl, precision)
    x, cond, t, lens = gl["x"].to(dev), gl["cond"].to(dev), gl["t_vec"], gl["lens_vec"]
    y2 = net(x, cond, t, lens_info=lens).cpu()
    for b in range(2):
        yb = net(x[b:b + 1], cond[b:b + 1], t[b:b + 1], lens_info=[v[b:b + 1] for v in lens]).cpu()
        assert torch.equal(y2[b:b + 1], yb), b
    sde = _sde(lib, gl, net, gl["cond"])
    sde.rng, sde.seed, sde.seed_auto_increment = "philox", 7, False
    xT = gl["x"].to(dev)
    sde.image_base = 0
    c2 = sde.reverse_sde(xT, lens_info=lens).cpu()
    for b in range(2):
        sde.set_mu(gl["cond"][b:b + 1].to(dev))
        sde.image_base = b
        cb = sde.reverse_sde(xT[b:b + 1], lens_info=[v[b:b + 1] for v in lens]).cpu()
        assert torch.isfinite(cb).all() and torch.equal(c2[b:b + 1], cb), b


def test_lens_change_on_one_plan(lib, gl):
    """Chains on one plan (same shape, same captured graph) with lens A, then lens B, then per-image lens each equal a fresh
    module's chain with that lens, bit for bit: the camera rows are re-written between chains and a change of the lens
    count (shared -> per image) re-captures the step graph."""
    dev = _dev()
    ch = gl["chain"]
    g = torch.Generator().manual_seed(3)
    lq = torch.rand(2, 4, 18, 23, generator=g)
    xT = (lq + torch.randn(lq.shape, generator=g) * 0.2).to(dev)
    zs = torch.randn((ch["T"],) + tuple(lq.shape), generator=g).to(dev)
    lens_a = [-18.0, 160.0, 3.5]
    lens_b = [torch.tensor([160.0]), torch.tensor([-18.0]), torch.tensor([12.0])]
    lens_c = gl["lens_vec"]
    sde = _sde(lib, gl, _net(lib, gl, "fp32"), lq)
    runs = [sde.reverse_sde(xT, zs=zs, lens_info=lens).cpu() for lens in (lens_a, lens_b, lens_c)]
    assert not torch.equal(runs[0], runs[1]) and not torch.equal(runs[1], runs[2])
    for lens, got in zip((lens_a, lens_b, lens_c), runs):
        fresh = _sde(lib, gl, _net(lib, gl, "fp32"), lq)
        assert torch.equal(fresh.reverse_sde(xT, zs=zs, lens_info=lens).cpu(), got)


def test_lens_errors(lib, gl):
    """Missing lens_info -> KeyError, wrong length -> ValueError, lens count neither 1 nor B -> IRSDE_ERR_INVALID; at the C
    ABI a lens network run before irsde_set_lens -> IRSDE_ERR_STATE, and irsde_set_lens on another network ->
    IRSDE_ERR_INVALID."""
    dev = _dev()
    net = _net(lib, gl, "fp32")
    x, cond = gl["x"].to(dev), gl["cond"].to(dev)
    with pytest.raises(KeyError, match="lens_info"):
        net(x, cond, 3)
    with pytest.raises(ValueError):
        net(x, cond, 3, lens_info=gl["lens_int"][:2])
    three = [torch.tensor([1.0, 2.0, 3.0])] * 3
    with pytest.raises(lib._lib.IrsdeError, match="batch size"):
        net(x, cond, 3, lens_info=three)
    fresh = _net(lib, gl, "fp32")
    ctx = fresh.sync_weights(dev)
    out = torch.empty_like(x)
    p = lambda a: ctypes.c_void_p(a.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = ctx.L.irsde_noise_fn(ctx.h, p(x), p(cond), lib._lib.float_array([3.0]), 1, p(out), 2, 18, 23, st)
    assert rc == -3  # IRSDE_ERR_STATE
    plain = lib.ConditionalNAFNet(**gl["cfg"]).to(dev)
    pctx = plain.sync_weights(dev)
    assert pctx.L.irsde_set_lens(pctx.h, lib._lib.float_array([1.0, 2.0, 3.0]), 1, st) == -1  # IRSDE_ERR_INVALID


def test_lens_bench_shape_bf16_vs_fp32(lib):
    """The bokeh YAML's network (w = 64, enc [2,2,4,8], mid 12, dec [2,2,2,2]) on one 1x4x360x480 latent (a 1440x1920
    image): bf16 vs fp32 on the device, both finite, within 4 % of scale (the oracle is too slow at this size)."""
    dev = _dev()
    cfg = dict(img_channel=4, width=64, middle_blk_num=12, enc_blk_nums=[2, 2, 4, 8], dec_blk_nums=[2, 2, 2, 2])
    P = L.make_nafnet_lens_weights(4, 64, 12, [2, 2, 4, 8], [2, 2, 2, 2], seed=9)
    for k in P:  # 36 residual blocks: keep the random residual branches at a trained network's scale
        if k.endswith("beta") or k.endswith("gamma"):
            P[k] = 0.2 * P[k]
    g = torch.Generator().manual_seed(10)
    lq = torch.rand(1, 4, 360, 480, generator=g).to(dev)
    x = lq + 0.3 * torch.randn(lq.shape, generator=g).to(dev)
    lens = [torch.tensor([-18.0]), torch.tensor([160.0]), torch.tensor([3.5])]
    ys = {}
    for prec in ("fp32", "bf16"):
        net = lib.ConditionalNAFNet(lens=True, precision=prec, **cfg)
        net.load_state_dict(P, strict=True)
        net = net.to(dev)
        ys[prec] = net(x, lq, 57, lens_info=lens).cpu()
        del net
        torch.cuda.empty_cache()
    assert torch.isfinite(ys["fp32"]).all() and torch.isfinite(ys["bf16"]).all()
    scale = ys["fp32"].abs().max().item()
    d = _maxdiff(ys["bf16"], ys["fp32"])
    print("bench shape: max|bf16 - fp32| = %.3e, scale %.3e" % (d, scale))
    assert scale > 0 and d <= 4e-2 * scale
