"""Drop-in launcher: run an UNMODIFIED reference script (codes/config/<task>/test.py, inference.py, ...)
on top of the B200-native sampler.

    python -m irsde_b200.run /path/to/codes/config/deraining/test.py -opt=options/test/ir-sde.yml

What it does before handing control to the script (nothing in the reference tree is edited):
  * chdir to the script's directory and reproduce its sys.path set-up (test.py:15-18 imports the
    cwd-local ``models``/``options`` and does ``sys.path.insert(0, "../../"); import utils``);
  * import the reference's ``utils`` package and swap ``IRSDE`` / ``DenoisingSDE`` for ours
    (codes/utils/sde_utils.py:80,373) - every other helper (img/file/deg utils) stays the reference's;
  * import the task's ``models.modules`` and swap ``ConditionalUNet`` for ours (the factory is
    ``getattr(M, which_model_G)(**setting)``, models/networks.py:10-15), choosing the variant by the
    reference class's own ``forward`` signature (``(x, time)`` => denoising-sde variant); likewise
    ``ConditionalNAFNet``: a ``forward`` taking ``**kwargs`` => the lens-conditioned latent-bokeh network
    (``lens=True``), otherwise ``latent=True`` when the task directory's name contains "latent";
  * provide tiny stand-ins for optional third-party modules the scripts import but this image lacks
    (IPython.embed, lpips.LPIPS, lmdb, ema_pytorch.EMA) - only when the real ones are not importable.

Precision / graph / RNG knobs come from the environment so existing YAMLs still parse:
IRSDE_B200_PRECISION=fp32|bf16|fp32x3, IRSDE_B200_GRAPH=0|1, IRSDE_B200_RNG=torch|philox.

Two launcher options (before the script path) exist for A/B parity runs (tests/test_gpu_dropin.py):
  --seed N       torch.manual_seed(N) right before the script starts (test.py never seeds: noise_state and the per-step
                 randn_like draws are otherwise irreproducible);
  --reference    do NOT swap anything: only the stand-ins for missing optional modules and the seed, i.e. the unmodified
                 reference on its own PyTorch path - the other arm of the comparison.
"""
import importlib
import inspect
import os
import runpy
import sys
import types


def _stub_missing():
    def have(name):
        try:
            importlib.import_module(name)
            return True
        except Exception:
            return False

    if not have("IPython"):
        m = types.ModuleType("IPython")
        m.embed = lambda *a, **k: None
        sys.modules["IPython"] = m
    if not have("lpips"):
        import torch

        class LPIPS(torch.nn.Module):  # metric only; needs AlexNet weights from the network
            def __init__(self, net="alex", **kw):
                super().__init__()

            def forward(self, a, b):
                return torch.zeros(1, device=a.device)

        m = types.ModuleType("lpips")
        m.LPIPS = LPIPS
        sys.modules["lpips"] = m
    if not have("lmdb"):
        sys.modules["lmdb"] = types.ModuleType("lmdb")
    if not have("ema_pytorch"):
        import torch

        class EMA(torch.nn.Module):
            def __init__(self, model, **kw):
                super().__init__()
                self.ema_model = model

            def update(self):
                pass

        m = types.ModuleType("ema_pytorch")
        m.EMA = EMA
        sys.modules["ema_pytorch"] = m


def install(script_dir):
    """Patch the reference packages reachable from ``script_dir`` (idempotent)."""
    import irsde_b200
    codes = os.path.abspath(os.path.join(script_dir, "..", ".."))
    for p in (script_dir, codes):
        if p not in sys.path:
            sys.path.insert(0, p)
    _stub_missing()
    utils = importlib.import_module("utils")
    utils.IRSDE = irsde_b200.IRSDE
    utils.DenoisingSDE = irsde_b200.DenoisingSDE
    if hasattr(utils, "sde_utils"):
        utils.sde_utils.IRSDE = irsde_b200.IRSDE
        utils.sde_utils.DenoisingSDE = irsde_b200.DenoisingSDE
    mods = importlib.import_module("models.modules")
    ref_cls = getattr(mods, "ConditionalUNet", None)
    ours = irsde_b200.ConditionalUNet
    if ref_cls is not None:
        params = list(inspect.signature(ref_cls.forward).parameters)
        if len(params) == 3:  # (self, x, time): denoising-sde variant
            ours = irsde_b200.DenoisingUNet
    mods.ConditionalUNet = ours
    if hasattr(mods, "ConditionalNAFNet"):
        import functools
        ref_naf = mods.ConditionalNAFNet
        if not (isinstance(ref_naf, functools.partial) or ref_naf is irsde_b200.ConditionalNAFNet):  # not installed yet
            kinds = [p.kind for p in inspect.signature(ref_naf.forward).parameters.values()]
            if inspect.Parameter.VAR_KEYWORD in kinds:  # forward(inp, cond, time, **kwargs): latent-bokeh's lens network
                mods.ConditionalNAFNet = functools.partial(irsde_b200.ConditionalNAFNet, lens=True)
            else:
                latent = "latent" in os.path.basename(os.path.abspath(script_dir))
                mods.ConditionalNAFNet = (functools.partial(irsde_b200.ConditionalNAFNet, latent=latent) if latent
                                          else irsde_b200.ConditionalNAFNet)
    if hasattr(mods, "UNet"):
        mods.UNet = irsde_b200.UNet
    return utils, mods


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    seed, reference = None, False
    while argv and argv[0].startswith("--"):
        opt = argv.pop(0)
        if opt == "--seed":
            seed = int(argv.pop(0))
        elif opt == "--reference":
            reference = True
        else:
            raise SystemExit("unknown launcher option %s\n%s" % (opt, __doc__))
    if not argv:
        raise SystemExit(__doc__)
    script = os.path.abspath(argv[0])
    script_dir = os.path.dirname(script)
    os.chdir(script_dir)
    if reference:
        codes = os.path.abspath(os.path.join(script_dir, "..", ".."))
        for p in (script_dir, codes):
            if p not in sys.path:
                sys.path.insert(0, p)
        _stub_missing()
    else:
        install(script_dir)
    if seed is not None:
        import torch
        torch.manual_seed(seed)
    sys.argv = [script] + argv[1:]
    runpy.run_path(script, run_name="__main__")


if __name__ == "__main__":
    main()
