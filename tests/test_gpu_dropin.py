"""Drop-in parity against the reference's own IRSDE + ConditionalUNet (SURVEY 8 b, f-4), held by a stored fixture
(tests/golden/reference_golden_dropin.pt, written by tests/golden/make_golden_dropin.py on a B200 from the reference's
classes driven the same way):
  * the native sampler driven the way the reference's `codes/config/deraining/test.py` drives it (test.py:67-72,93-110:
    noise_state on the CPU LQ tensor, set_mu, reverse_<mode>, tensor2img) reproduces the reference's output images to
    within one grey level (uint8 rounding of a <=1e-3 difference), for reverse_posterior and reverse_sde;
  * validation sampling during training (train.py:214-215,236,261-281) adopts a foreign PyTorch ConditionalUNet that keeps
    being trained by autograd, with its current weights before and after an optimizer step.
Both use the same seeded weights (oracle.make_weights) and the torch CUDA generator for the noise, which the native
sampler's torch-RNG mode draws in the reference's order."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_golden_dropin.pt")
SDE_ARGS = dict(max_sigma=10, T=12, schedule="cosine", eps=0.005)
NET_ARGS = (3, 3, 16, 2)   # in_nc, out_nc, nf, depth
SEED = 123


def weights():
    """Seeded weights; the final conv is scaled down so that outputs are of the size a default-initialised network gives."""
    from oracle import irsde_oracle as O
    return O.make_weights(*NET_ARGS, seed=0, out_gain=0.1)


def images():
    """Three (GT, LQ) uint8 BGR pairs; the last two sizes are not multiples of 4 (the UNet reflect-pads them)."""
    rng = np.random.RandomState(0)
    out = []
    for h, w in [(64, 64), (48, 80), (50, 38)]:
        gt = (rng.rand(h, w, 3) * 255).astype(np.uint8)
        lq = np.clip(gt.astype(np.int32) + rng.randint(-30, 30, gt.shape), 0, 255).astype(np.uint8)
        out.append((gt, lq))
    return out


def to_tensor(img):
    """uint8 HWC BGR -> float32 1x3xHxW RGB in [0, 1], as the reference's LQGT dataset hands images to test.py."""
    import torch
    x = img.astype(np.float32) / 255.0
    return torch.from_numpy(np.ascontiguousarray(x[:, :, [2, 1, 0]].transpose(2, 0, 1)))[None]


def foreign_unet(P):
    """A plain PyTorch module with the reference ConditionalUNet's state-dict layout whose forward is the oracle's:
    stands in for the reference's own class being trained by autograd.  The forward runs on the host (the oracle is
    CPU code); gradients flow back to the parameters on the device."""
    import torch
    from oracle import irsde_oracle as O

    class ForeignUNet(torch.nn.Module):
        def forward(self, xt, cond, time):
            p = {k: v.cpu() for k, v in self.named_parameters()}
            t = time.cpu() if torch.is_tensor(time) else time
            return O.unet_forward(p, xt.cpu(), cond.cpu(), t, NET_ARGS[2], NET_ARGS[3]).to(xt.device)

    root = ForeignUNet()
    for name, v in P.items():
        *path, leaf = name.split(".")
        m = root
        for p in path:
            if p not in m._modules:
                m.add_module(p, torch.nn.Module())
            m = m._modules[p]
        m.register_parameter(leaf, torch.nn.Parameter(v.clone()))
    assert list(root.state_dict().keys()) == list(P.keys())
    return root


@pytest.mark.parametrize("mode", ["posterior", "sde"])
def test_test_py_sampling_matches_reference_images(mode):
    import torch
    import irsde_b200
    from oracle import imaging_oracle as IO
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    gold = torch.load(GOLDEN, weights_only=True)["test_py"][mode]
    dev = torch.device("cuda:0")
    net = irsde_b200.ConditionalUNet(*NET_ARGS[:3], depth=NET_ARGS[3], precision="fp32")
    net.load_state_dict(weights(), strict=True)
    net = net.to(dev)
    sde = irsde_b200.IRSDE(device=dev, **SDE_ARGS)
    sde.set_model(net)
    torch.manual_seed(SEED)
    worst = 0
    for (gt, lq), ref in zip(images(), gold):
        LQ, GT = to_tensor(lq), to_tensor(gt)
        noisy = sde.noise_state(LQ)
        sde.set_mu(LQ.to(dev))
        with torch.no_grad():
            out = getattr(sde, "reverse_" + mode)(noisy.to(dev))
        img = IO.tensor2img(out[0].float().cpu().numpy())
        assert img.shape == tuple(ref.shape)
        worst = max(worst, int(np.abs(img.astype(np.int32) - ref.numpy().astype(np.int32)).max()))
        # the reference wrote its _LQ / _HQ images back bit for bit (checked when the fixture was made)
        assert np.array_equal(IO.tensor2img(LQ[0].numpy()), lq) and np.array_equal(IO.tensor2img(GT[0].numpy()), gt)
    assert worst <= 1, "restored images differ by %d grey levels" % worst
    assert net.launch_count() > 0


def test_validation_sampling_adopts_reference_module_during_training():
    """SURVEY 8 f-4 (train.py:214-215,236,261-281): a PyTorch ConditionalUNet keeps being trained by autograd;
    `sde.set_model(DataParallel(net))` + `model.eval()` + `sde.reverse_posterior(...)` must sample through the native
    kernels with the module's CURRENT weights (before and after an optimizer step), and `generate_random_states` must give
    the reference's states bit for bit."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import irsde_b200
    gold = torch.load(GOLDEN, weights_only=True)["training"]
    dev = torch.device("cuda:0")
    ref_net = foreign_unet(weights()).to(dev)
    wrapped = torch.nn.DataParallel(ref_net, device_ids=[0])
    ours = irsde_b200.IRSDE(device=dev, **SDE_ARGS)
    ours.set_model(wrapped)
    g = torch.Generator().manual_seed(1)
    GT, LQ = torch.rand(2, 3, 24, 40, generator=g), torch.rand(2, 3, 24, 40, generator=g)

    # ---- train.py:236  generate_random_states: same generator calls, bit-identical states
    torch.manual_seed(5)
    t_our, s_our = ours.generate_random_states(x0=GT, mu=LQ)
    assert torch.equal(gold["t"], t_our.cpu()) and torch.equal(gold["states"], s_our.cpu())

    opt = torch.optim.SGD(ref_net.parameters(), lr=1e-2)

    def validate():
        wrapped.eval()
        ours.set_mu(LQ.to(dev))
        torch.manual_seed(9)
        with torch.no_grad():
            out = ours.reverse_posterior(LQ.to(dev) + 0.03)
        wrapped.train()
        return out.cpu()

    a_our = validate()
    assert (gold["a"] - a_our).abs().max().item() < 1e-3
    shadow = getattr(ref_net, "_irsde_b200_shadow", None)
    assert shadow is not None and shadow is not False and shadow.launch_count() > 0     # the native kernels ran
    # ---- one real training step through the module's autograd forward (train.py:239 optimize_parameters)
    ref_net.train()
    torch.manual_seed(11)   # the training batch must not depend on how many numbers validation drew (shadow set-up included)
    ts, states = ours.generate_random_states(x0=GT, mu=LQ)
    noise = ours.noise_fn(states, ts.squeeze().to(dev))
    loss = noise.pow(2).mean()
    loss.backward()
    opt.step()
    b_our = validate()
    assert (gold["b"] - b_our).abs().max().item() < 1e-3           # the shadow picked up the updated weights
    assert (gold["b"] - gold["a"]).abs().max().item() > 1e-4       # and the step did change the result
