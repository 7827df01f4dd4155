"""CPU tests of the lens-conditioned ConditionalNAFNet (latent-bokeh): the oracle against the reference's own outputs, the
state-dict contract, argument checks that run before any device work, the sampler's fast-path rule and the launcher rule."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from oracle import irsde_oracle as O  # noqa: E402
import _lens_oracle as L  # noqa: E402


@pytest.fixture(scope="module")
def gl():
    return torch.load(os.path.join(ROOT, "tests", "golden", "reference_golden_lens.pt"), weights_only=True)


def _args(c):
    return c["width"], c["enc_blk_nums"], c["middle_blk_num"], c["dec_blk_nums"]


def test_lens_oracle_vs_reference(gl):
    """Forwards (B = 1 with int t and 1-element lens tensors; B = 2 with per-image t and lens) <= 1e-5 and the reference's
    own IRSDE.reverse_sde(..., lens_info=...) chain (T = 8, replayed z) <= 2e-4."""
    c = gl["cfg"]
    y = L.nafnet_lens_forward(gl["state"], gl["x"][:1], gl["cond"][:1], gl["t_int"], gl["lens_int"], *_args(c))
    assert (y - gl["y_int"]).abs().max().item() <= 1e-5
    yv = L.nafnet_lens_forward(gl["state"], gl["x"], gl["cond"], gl["t_vec"], gl["lens_vec"], *_args(c))
    assert (yv - gl["y_vec"]).abs().max().item() <= 1e-5
    ch = gl["chain"]
    sc = O.Schedule(ch["max_sigma"], ch["T"], "cosine", ch["eps"])
    fn = lambda x, t: L.nafnet_lens_forward(gl["state"], x, ch["lq"], t, ch["lens"], *_args(c))
    x0 = O.reverse_chain(sc, fn, ch["xT"], ch["lq"], ch["zs"], "sde")
    assert (x0 - ch["x0"]).abs().max().item() <= 2e-4
    shapes = L.nafnet_lens_param_shapes(c["img_channel"], c["width"], c["middle_blk_num"], c["enc_blk_nums"],
                                        c["dec_blk_nums"])
    assert list(shapes) == list(gl["state"]) and all(tuple(gl["state"][k].shape) == tuple(v) for k, v in shapes.items())


def test_lens_state_dict_contract(gl):
    """ConditionalNAFNet(lens=True) registers exactly the reference's keys, shapes and order and strict-loads them."""
    import irsde_b200
    net = irsde_b200.ConditionalNAFNet(lens=True, **gl["cfg"])
    sd = net.state_dict()
    assert list(sd.keys()) == list(gl["state"].keys())
    assert all(tuple(sd[k].shape) == tuple(v.shape) for k, v in gl["state"].items())
    net.load_state_dict(gl["state"], strict=True)
    c = gl["cfg"]
    assert irsde_b200.nafnet_param_shapes(c["img_channel"], c["width"], c["middle_blk_num"], c["enc_blk_nums"],
                                          c["dec_blk_nums"], lens=True) == \
        {k: tuple(v) for k, v in L.nafnet_lens_param_shapes(c["img_channel"], c["width"], c["middle_blk_num"],
                                                            c["enc_blk_nums"], c["dec_blk_nums"]).items()}
    with pytest.raises(ValueError):
        irsde_b200.ConditionalNAFNet(lens=True, latent=True, **c)


def test_lens_argument_checks_before_device_work(gl):
    """Missing lens_info raises KeyError('lens_info') as the reference does; a lens_info that is not 3 entries, or whose
    entries disagree in length, raises ValueError; the non-lens variants still reject keyword arguments."""
    import irsde_b200
    net = irsde_b200.ConditionalNAFNet(lens=True, **gl["cfg"])
    x = gl["x"][:1]
    with pytest.raises(KeyError, match="lens_info"):
        net(x, x, 3)
    with pytest.raises(ValueError):
        net(x, x, 3, lens_info=[1.0, 2.0])
    with pytest.raises(ValueError):
        net(x, x, 3, lens_info=[torch.tensor([1.0, 2.0]), torch.tensor([1.0, 2.0, 3.0]), 0.5])
    rows = irsde_b200.ConditionalNAFNet.lens_rows([torch.tensor([-18.0]), 160, torch.tensor([3.5], dtype=torch.float64)])
    assert rows.dtype == torch.float32 and rows.tolist() == [[-18.0, 160.0, 3.5]]
    rows = irsde_b200.ConditionalNAFNet.lens_rows([torch.tensor([-18.0, 18.0]), 160.0, torch.tensor([3.5, 12.0])])
    assert rows.tolist() == [[-18.0, 160.0, 3.5], [18.0, 160.0, 12.0]]
    plain = irsde_b200.ConditionalNAFNet(**gl["cfg"])
    with pytest.raises(TypeError):
        plain(x, x, 3, lens_info=[1.0, 2.0, 3.0])


def test_sampler_fast_path_rule(gl):
    """IRSDE runs the whole chain natively for a lens network only when the one keyword is lens_info; a lens network without
    it takes the per-step loop (which raises the reference's KeyError); other networks keep taking no keywords."""
    import irsde_b200
    sde = irsde_b200.IRSDE(50, 8, schedule="cosine", eps=0.005, device="cpu")
    sde.set_model(irsde_b200.ConditionalNAFNet(lens=True, **gl["cfg"]))
    lens = {"lens_info": [1.0, 2.0, 3.0]}
    assert sde._fast(lens, False) and not sde._fast({}, False) and not sde._fast(lens, True)
    assert not sde._fast(dict(lens, other=1), False)
    sde.set_model(irsde_b200.ConditionalNAFNet(**gl["cfg"]))
    assert sde._fast({}, False) and not sde._fast(lens, False)


def _tree(root, task, naf_forward):
    files = {
        "codes/utils/__init__.py": "from .sde_utils import *\n",
        "codes/utils/sde_utils.py": "class IRSDE:\n    pass\n\n\nclass DenoisingSDE:\n    pass\n",
        "codes/config/%s/models/__init__.py" % task: "",
        "codes/config/%s/models/networks.py" % task: (
            "from models import modules as M\n\n\n"
            "def define_G(opt):\n"
            "    net = opt['network_G']\n"
            "    return getattr(M, net['which_model_G'])(**net['setting'])\n"),
        "codes/config/%s/models/modules/__init__.py" % task: (
            "import torch\n\n\n"
            "class ConditionalUNet(torch.nn.Module):\n"
            "    def forward(self, xt, cond, time):\n"
            "        raise AssertionError('the PyTorch network must not be used')\n\n\n"
            "class ConditionalNAFNet(torch.nn.Module):\n"
            "    def forward(%s):\n"
            "        raise AssertionError('the PyTorch network must not be used')\n" % naf_forward),
    }
    for rel, text in files.items():
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(text)
    return os.path.join(root, "codes", "config", task)


@pytest.mark.parametrize("task,forward,lens,latent", [
    ("latent-bokeh", "self, inp, cond, time, **kwargs", True, False),
    ("latent-dehazing", "self, inp, cond, time", False, True),
])
def test_launcher_picks_nafnet_variant(tmp_path, task, forward, lens, latent):
    """`run.install` picks the lens network when the reference ConditionalNAFNet.forward takes **kwargs (latent-bokeh), and
    keeps the directory-name rule for `latent` otherwise."""
    ref = _tree(str(tmp_path), task, forward)
    code = (
        "import sys, os; sys.path.insert(0, %r); import irsde_b200; from irsde_b200 import run; os.chdir(%r); "
        "u, m = run.install(%r); run.install(%r); from models import networks; "
        "naf = networks.define_G({'network_G': {'which_model_G': 'ConditionalNAFNet', 'setting': dict(img_channel=4, width=8, "
        "enc_blk_nums=[1], middle_blk_num=1, dec_blk_nums=[1])}}); "
        "assert isinstance(naf, irsde_b200.ConditionalNAFNet); print('variant', naf.lens, naf.latent)" % (ROOT, ref, ref, ref))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "variant %s %s" % (lens, latent) in out.stdout
