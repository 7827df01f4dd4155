"""CPU-side tests: C-ABI exports, host logic (schedules, state-dict contract, sharding plumbing)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import irsde_b200
    L = irsde_b200._lib.load()
    hdr = open(os.path.join(ROOT, "include", "irsde_b200.h")).read()
    declared = set(re.findall(r"\b(irsde_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(irsde_b200._lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s
    assert b"sm_100a" in L.irsde_version()


def test_no_gpu_fails_loudly():
    import irsde_b200
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(irsde_b200._lib.IrsdeError):
        irsde_b200._lib.Context(3, 3, 8, 2, 0, 0, 0)
    net = irsde_b200.ConditionalUNet(3, 3, 8, depth=2)
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 3, 8, 8), torch.zeros(1, 3, 8, 8), 1)


def test_state_dict_contract(golden):
    import irsde_b200
    for key, cls in (("unet_cond", irsde_b200.ConditionalUNet), ("unet_dsde", irsde_b200.DenoisingUNet)):
        g = golden[key]
        net = cls(3, 3, g["nf"], depth=g["depth"])
        assert list(net.state_dict().keys()) == list(g["state"].keys())
        net.load_state_dict(g["state"], strict=True)
        wrapped = torch.nn.DataParallel(net) if torch.cuda.is_available() else net
        assert irsde_b200.sde._unwrap(wrapped) is net


def test_schedule_tables_match_reference(golden):
    import irsde_b200
    for g in golden["irsde_schedules"]:
        ms, T, s, eps = g["args"]
        sde = irsde_b200.IRSDE(ms, T, schedule=s, eps=eps, device="cpu")
        for k in ("thetas", "sigmas", "thetas_cumsum", "sigma_bars"):
            assert torch.equal(getattr(sde, k), g[k])
        assert torch.equal(torch.as_tensor(sde.dt), g["dt"])
    for g in golden["dsde_schedules"]:
        ms, T, s = g["args"]
        sde = irsde_b200.DenoisingSDE(ms, T, schedule=s, device="cpu")
        assert torch.equal(sde.sigma_bars, g["sigma_bars"])
        for sg, t in g["optimal_t"].items():
            assert int(sde.get_optimal_timestep(sg)) == t


def test_coeff_tables_reproduce_reference_steps(golden):
    """The [T+1][8] scalar tables + the kernel's formula (restated in torch) give the reference step."""
    import irsde_b200
    L = irsde_b200._lib
    g = golden["irsde_steps"]
    sde = irsde_b200.IRSDE(g["args"][0], g["args"][1], schedule=g["args"][2], eps=g["args"][3], device="cpu")
    x, mu, eps_ = g["x"], g["mu"], g["noise"]
    for st in g["steps"]:
        t, z = st["t"], st["z"]
        c = sde._coeff_table(L.MODE_SDE)[t]
        out = x - ((c[0] * (mu - x) - c[1] * (-eps_ / c[2])) * c[3]) - c[4] * (z * c[5])
        assert torch.equal(out, st["sde"])
        c = sde._coeff_table(L.MODE_POSTERIOR)[t]
        x0 = (x - mu - c[1] * eps_) * c[0] + mu
        out = c[2] * (x - mu) + c[3] * (x0 - mu) + mu + c[4] * z
        assert torch.equal(out, st["posterior"])


def test_shard_range_partition():
    import irsde_b200
    for B in (1, 3, 8, 32, 33):
        for R in (1, 2, 4, 8):
            cover = []
            for r in range(R):
                lo, hi = irsde_b200.shard_range(B, r, R)
                cover += list(range(lo, hi))
            assert cover == list(range(B))


def _worker(rank, world, port, q):
    import torch.distributed as dist
    import irsde_b200
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    xT = torch.arange(5 * 3 * 2 * 2, dtype=torch.float32).reshape(5, 3, 2, 2)
    mu = xT * 0.5
    zs = torch.arange(4 * 5 * 3 * 2 * 2, dtype=torch.float32).reshape(4, 5, 3, 2, 2)
    run = lambda x, m, z: x * 2 + m + z.sum(0)  # stand-in for the per-rank chain (needs no GPU)
    out = irsde_b200.sharded_reverse(run, xT, mu, zs)

    class FakeSde:  # in-kernel Philox path: the rank's first global image index must be the image base during the run
        image_base = 100
    seen = []
    run2 = lambda x, m, z: (seen.append((FakeSde.image_base, x.shape[0], z is None)), x + 1)[1]
    out2 = irsde_b200.sharded_reverse(run2, xT, mu, None, sde=FakeSde)
    lo, hi = irsde_b200.shard_range(5, rank, world)
    assert seen == [(100 + lo, hi - lo, True)] and FakeSde.image_base == 100 and torch.equal(out2, xT + 1)
    lin = torch.nn.Linear(4, 4)
    if rank != 0:
        with torch.no_grad():
            for p in lin.parameters():
                p.zero_()
    irsde_b200.broadcast_weights(lin, src=0)
    # numpy payloads are pickled by value; a tensor travels as a shared-memory fd that dies with this worker (flaky)
    q.put((rank, out.numpy(), torch.cat([p.detach().reshape(-1) for p in lin.parameters()]).numpy()))
    dist.destroy_process_group()


def test_sharded_gather_gloo_world2():
    """world_size=2 gloo: partition, per-rank run, all_gather order, one-shot weight broadcast."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted([q.get(timeout=120) for _ in ps], key=lambda r: r[0])
    res = [(r, torch.from_numpy(o), torch.from_numpy(w)) for r, o, w in res]
    for p in ps:
        p.join(60)
    xT = torch.arange(5 * 3 * 2 * 2, dtype=torch.float32).reshape(5, 3, 2, 2)
    zs = torch.arange(4 * 5 * 3 * 2 * 2, dtype=torch.float32).reshape(4, 5, 3, 2, 2)
    expect = xT * 2 + xT * 0.5 + zs.sum(0)
    for rank, out, w in res:
        assert torch.equal(out, expect)
    assert torch.equal(res[0][2], res[1][2]) and res[0][2].abs().sum() > 0


def _reference_layout_tree(root):
    """A minimal tree with the reference's package layout as the launcher sees it: `codes/utils` re-exports the samplers
    of `utils/sde_utils.py`; `codes/config/deraining/models/networks.py` builds the network with
    `getattr(models.modules, which_model_G)(**setting)` (networks.py:10-15); `models.modules` exports the PyTorch
    ConditionalUNet (forward(xt, cond, time)) and ConditionalNAFNet."""
    files = {
        "codes/utils/__init__.py": "from .sde_utils import *\n",
        "codes/utils/sde_utils.py": "class IRSDE:\n    pass\n\n\nclass DenoisingSDE:\n    pass\n",
        "codes/config/deraining/models/__init__.py": "",
        "codes/config/deraining/models/networks.py": (
            "from models import modules as M\n\n\n"
            "def define_G(opt):\n"
            "    net = opt['network_G']\n"
            "    return getattr(M, net['which_model_G'])(**net['setting'])\n"),
        "codes/config/deraining/models/modules/__init__.py": (
            "import torch\n\n\n"
            "class ConditionalUNet(torch.nn.Module):\n"
            "    def forward(self, xt, cond, time):\n"
            "        raise AssertionError('the PyTorch network must not be used')\n\n\n"
            "class ConditionalNAFNet(ConditionalUNet):\n"
            "    pass\n"),
    }
    for rel, text in files.items():
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(text)
    return os.path.join(root, "codes", "config", "deraining")


def test_launcher_patches_reference_tree(tmp_path):
    """Drop-in mechanics (INTEGRATION.md 1): on a tree laid out like the reference's, `run.install` swaps the sampler and
    network classes the reference scripts resolve by name."""
    ref = _reference_layout_tree(str(tmp_path))
    import subprocess
    import sys
    code = (
        "import sys, os; sys.path.insert(0, %r); import irsde_b200; from irsde_b200 import run; os.chdir(%r); "
        "u, m = run.install(%r); from models import networks; "
        "assert u.IRSDE is irsde_b200.IRSDE and u.DenoisingSDE is irsde_b200.DenoisingSDE; "
        "net = networks.define_G({'network_G': {'which_model_G': 'ConditionalUNet', 'setting': dict(in_nc=3, out_nc=3, nf=8, depth=2)}}); "
        "assert isinstance(net, irsde_b200.ConditionalUNet); "
        "naf = networks.define_G({'network_G': {'which_model_G': 'ConditionalNAFNet', 'setting': dict(img_channel=3, width=8, enc_blk_nums=[1], middle_blk_num=1, dec_blk_nums=[1])}}); "
        "assert isinstance(naf, irsde_b200.ConditionalNAFNet); print('ok')" % (ROOT, ref, ref))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_plan_batches_groups_by_shape():
    import irsde_b200
    shapes = [(4, 4, 3), (8, 8, 3), (4, 4, 3), (4, 4, 3), (8, 8, 3), (4, 4, 3)]
    plan = irsde_b200.plan_batches(shapes, 2)
    assert plan == [((4, 4, 3), [0, 2]), ((4, 4, 3), [3, 5]), ((8, 8, 3), [1, 4])]
    assert sorted(i for _, idx in plan for i in idx) == list(range(6))           # every image exactly once
    assert irsde_b200.plan_batches([], 4) == []
    import pytest
    with pytest.raises(ValueError):
        irsde_b200.plan_batches(shapes, 0)


def test_sde_diagnostic_helpers_match_reference_algebra():
    """drift / reverse drifts / reverse_optimum_std / forward_step: the reference's formulas (sde_utils.py:170-182,207-217,
    446-456) evaluated on CPU tensors - these helpers are plain tensor algebra and need no GPU."""
    import math
    import torch
    import irsde_b200
    sde = irsde_b200.IRSDE(max_sigma=30, T=20, schedule="cosine", eps=0.005, device="cpu")
    g = torch.Generator().manual_seed(0)
    x, mu, sc = (torch.randn(2, 3, 4, 4, generator=g) for _ in range(3))
    sde.set_mu(mu)
    t = 7
    th, sg, dt = sde.thetas[t], sde.sigmas[t], sde.dt
    assert torch.equal(sde.drift(x, t), th * (mu - x) * dt)
    assert torch.equal(sde.sde_reverse_drift(x, sc, t), (th * (mu - x) - sg ** 2 * sc) * dt)
    assert torch.equal(sde.ode_reverse_drift(x, sc, t), (th * (mu - x) - 0.5 * sg ** 2 * sc) * dt)
    assert torch.equal(sde.reverse_sde_step_mean(x, sc, t), x - sde.sde_reverse_drift(x, sc, t))
    torch.manual_seed(3)
    d = sde.dispersion(x, t)
    torch.manual_seed(3)
    assert torch.equal(d, sg * (torch.randn_like(x) * math.sqrt(dt)))
    # posterior std equals the closed form and collapses at t = 1 (deterministic last step, SURVEY 8 a-6)
    A, B, C = (torch.exp(-2 * v * dt) for v in (sde.thetas[t], sde.thetas_cumsum[t], sde.thetas_cumsum[t - 1]))
    assert abs(sde.reverse_optimum_std(t).item() - (((1 - A) * (1 - C) / (1 - B)).sqrt() * sde.max_sigma).item()) < 1e-7
    assert sde.reverse_optimum_std(1).item() < 1e-9
    # optimal_reverse with the true x0 walks back to x0
    x0 = torch.rand(1, 3, 4, 4, generator=g)
    sde.set_mu(torch.rand(1, 3, 4, 4, generator=g))
    xT = sde.mu_bar(x0, sde.T)
    assert (sde.optimal_reverse(xT, x0) - x0).abs().max().item() < 1e-3
    ds = irsde_b200.DenoisingSDE(max_sigma=50, T=20, device="cpu")
    Ad = torch.exp(-2 * ds.thetas_cumsum[t] * ds.dt)
    assert torch.equal(ds.sde_reverse_drift(x, sc, t), -0.5 * ds.sigmas[t] ** 2 * (1 + Ad) * sc * ds.dt)
    assert torch.equal(ds.ode_reverse_drift(x, sc, t), -0.5 * ds.sigmas[t] ** 2 * Ad * sc * ds.dt)
    assert torch.equal(ds.drift(x, mu, t), ds.thetas[t] * (mu - x) * ds.dt)


def test_state_dict_contract_nafnet_and_latent():
    """ConditionalNAFNet (both variants) and the latent UNet register exactly the reference's state-dict keys/shapes
    (fixtures hold the reference modules' own state_dict), so `load_state_dict(strict=True)` of reference checkpoints works."""
    import irsde_b200
    gd = os.path.join(os.path.dirname(__file__), "golden")
    naf = torch.load(os.path.join(gd, "reference_golden_nafnet.pt"), weights_only=True)
    for key, g in naf.items():
        if not (isinstance(g, dict) and "state" in g):
            continue
        net = irsde_b200.ConditionalNAFNet(latent=g["latent"], **g["cfg"])
        assert list(net.state_dict().keys()) == list(g["state"].keys()), key
        assert all(tuple(net.state_dict()[k].shape) == tuple(v.shape) for k, v in g["state"].items())
        net.load_state_dict(g["state"], strict=True)
    lat = torch.load(os.path.join(gd, "reference_golden_latent.pt"), weights_only=True)
    ae = irsde_b200.UNet(**lat["cfg"])
    assert list(ae.state_dict().keys()) == list(lat["state"].keys())
    ae.load_state_dict(lat["state"], strict=True)
    from oracle import irsde_oracle as O
    c = lat["cfg"]
    assert irsde_b200.latent_unet_param_shapes(c["in_ch"], c["out_ch"], c["ch"], c["ch_mult"], c["embed_dim"]) == \
        {k: tuple(v) for k, v in O.latent_unet_param_shapes(c["in_ch"], c["out_ch"], c["ch"], c["ch_mult"], c["embed_dim"]).items()}


def test_front_end_needs_cuda():
    """imaging / Restorer / latent UNet have no CPU path: they raise instead of silently computing on the host."""
    import numpy as np
    import irsde_b200
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    img = np.zeros((16, 16, 3), np.uint8)
    with pytest.raises(RuntimeError):
        irsde_b200.tensor2img(torch.zeros(3, 16, 16))
    with pytest.raises(RuntimeError):
        irsde_b200.calculate_psnr(img, img)
    with pytest.raises(RuntimeError):
        irsde_b200.UNet(3, 3, 8, [1, 2], 4).encode(torch.zeros(1, 3, 16, 16))
    sde = irsde_b200.IRSDE(10, 4, device="cpu")
    with pytest.raises(RuntimeError):
        irsde_b200.Restorer(sde, device="cpu").restore([img])
    with pytest.raises(TypeError):
        irsde_b200.Restorer(sde, device="cpu").restore([img.astype(np.float32)])


# ---- Refusion tile sharding: host logic (grid, grouping by shape, unit partition, gathers, stitching) on gloo ------------
class _FakeAE:
    """CPU stand-in for the latent autoencoder: 'encode' = 2x2 average pool of 4 channels, 'decode' = nearest upsample."""
    def encode(self, x):
        z = torch.nn.functional.avg_pool2d(torch.cat([x, x[:, :1]], 1), 2)
        return z, ("skips", x.shape)

    def decode(self, z, h):
        assert h[0] == "skips" and h[1][0] == z.shape[0]
        return torch.nn.functional.interpolate(z[:, :3], scale_factor=2, mode="nearest")


def _fake_chain(mu, uids):   # depends on the tile content AND the unit's global uid AND the tile's own mean (a "global" op)
    u = torch.tensor(uids, dtype=torch.float32)[:, None, None, None]
    return mu * 2 + u + mu.mean(dim=(2, 3), keepdim=True)


def _tile_worker(rank, world, port, q):
    import torch.distributed as dist
    import irsde_b200
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    LQ = torch.arange(3 * 3 * 20 * 28, dtype=torch.float32).reshape(3, 3, 20, 28) / 100.0
    tr = irsde_b200.TiledRefusion(_FakeAE(), None, tile=4, chain=_fake_chain)   # latent 10x14 -> 3x4 grid, ragged edges
    out, (lo, hi) = tr.restore(LQ)
    q.put((rank, lo, hi, out.numpy()))   # numpy: pickled by value (a tensor's shared-memory fd dies with the worker)
    dist.destroy_process_group()


def test_tile_grid_and_units():
    import irsde_b200
    assert irsde_b200.tile_boxes(10, 14, 4) == [(y, min(y + 4, 10), x, min(x + 4, 14)) for y in (0, 4, 8) for x in (0, 4, 8, 12)]
    assert irsde_b200.tile_boxes(10, 14, None) == [(0, 10, 0, 14)]
    units, groups = irsde_b200.plan_units(2, 10, 14, 4)
    assert [u[0] for u in units] == list(range(24)) and units[13][1] == 1
    assert sorted(groups) == [(2, 2), (2, 4), (4, 2), (4, 4)]
    assert sum(len(v) for v in groups.values()) == 24 and len(groups[(4, 4)]) == 12
    cover = torch.zeros(10, 14)
    for _, b, (y0, y1, x0, x1) in units[:12]:
        cover[y0:y1, x0:x1] += 1
    assert (cover == 1).all()           # tiles partition the latent: every pixel exactly once


@pytest.mark.parametrize("world", [2, 4])
def test_tiled_refusion_gloo(world):
    """world_size 2 and 4 (4 ranks > 3 images: one rank owns no image but still processes tiles): the sharded pipeline
    reproduces the single-process result exactly, and that equals the per-tile definition computed by hand."""
    import torch.multiprocessing as mp
    import irsde_b200
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() + world) % 2000
    ps = [ctx.Process(target=_tile_worker, args=(r, world, port, q)) for r in range(world)]
    for p in ps:
        p.start()
    res = sorted([q.get(timeout=120) for _ in ps], key=lambda r: r[0])
    for p in ps:
        p.join(60)
    LQ = torch.arange(3 * 3 * 20 * 28, dtype=torch.float32).reshape(3, 3, 20, 28) / 100.0
    single, _ = irsde_b200.TiledRefusion(_FakeAE(), None, tile=4, chain=_fake_chain).restore(LQ)
    got = torch.cat([torch.from_numpy(r[3]) for r in res])
    assert [(r[1], r[2]) for r in res] == [irsde_b200.shard_range(3, r, world) for r in range(world)]
    assert torch.equal(got, single)
    # by hand: every tile independently, uid = image * tiles_per_image + tile index
    ae = _FakeAE()
    z, h = ae.encode(LQ)
    ref = torch.empty_like(z)
    boxes = irsde_b200.tile_boxes(10, 14, 4)
    for b in range(3):
        for k, (y0, y1, x0, x1) in enumerate(boxes):
            ref[b:b + 1, :, y0:y1, x0:x1] = _fake_chain(z[b:b + 1, :, y0:y1, x0:x1], [b * len(boxes) + k])
    assert torch.allclose(single, ae.decode(ref, h), rtol=1e-6, atol=1e-4)   # batch-of-tiles vs one-tile reductions: last ulp


def test_ncu_summariser_refuses_a_capture_without_the_shipped_kernels(tmp_path):
    """scripts/ncu_summarize.py --require: the round-1 profiles described a kernel that was no longer the shipped one; the
    summariser now fails (exit 3) unless every required kernel-name pattern occurs, and records the kernel mix."""
    import json
    import subprocess
    import sys
    raw = tmp_path / "raw.csv"
    raw.write_text('"ID","Kernel Name","Grid Size","gpu__time_duration.sum"\n"","","","us"\n'
                   '"0","void irsde::<unnamed>::conv_tc_persist_kernel<(int)64, (int)2, (int)1, (int)6>(CUtensorMap_st)","(148, 1, 1)","10"\n'
                   '"1","void irsde::<unnamed>::conv_tc_persist_kernel<(int)256, (int)0, (int)2, (int)12>(CUtensorMap_st)","(148, 1, 1)","20"\n')
    script = os.path.join(ROOT, "scripts", "ncu_summarize.py")
    ok = subprocess.run([sys.executable, script, str(raw), "--require", r"conv_tc_persist_kernel<\d+, 2[,>]", "--meta",
                         str(tmp_path / "m.json"), "commit=abc"], capture_output=True, text=True)
    assert ok.returncode == 0 and "gpu__time_duration.sum" in ok.stdout
    meta = json.load(open(tmp_path / "m.json"))
    assert meta["commit"] == "abc" and meta["kernel_mix"] == {"conv_tc_persist_kernel<64, 2, 1, 6>": 1, "conv_tc_persist_kernel<256, 0, 2, 12>": 1}
    bad = subprocess.run([sys.executable, script, str(raw), "--require", r"conv_tc_persist_kernel<\d+, 3[,>]"], capture_output=True, text=True)
    assert bad.returncode == 3 and "no kernel matches" in bad.stderr


def test_committed_conv_capture_is_of_the_shipped_conv_kernel_sources():
    """The roofline's `traffic` comes from profiles/r*_conv_tc_ncu_full_one_step.csv: its .meta.json names the hash of the
    sources the tcgen05 conv kernel compiles from (conv_tc.cu + common.cuh).  Changing the conv kernel without re-capturing
    fails here (round 1 shipped a capture of a kernel that was no longer the benchmarked one)."""
    import glob
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("irsde_build", os.path.join(ROOT, "image-restoration-sde_b200", "build.py"))
    build = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(build)
    metas = sorted(m for m in glob.glob(os.path.join(ROOT, "profiles", "r*_conv_tc_ncu_full_one_step.meta.json")) if "_v1_" not in m)
    assert metas, "no committed conv capture"
    meta = json.load(open(metas[-1]))
    assert meta["conv_tc_sha256"] == build.conv_tc_sha256()
    mix = meta["kernel_mix"]
    assert any(re.match(r"conv_tc_persist_kernel<\d+, 2,", k) for k in mix) and any(k.startswith("conv_tc_persist_kernel<256, 0, 2") for k in mix)
