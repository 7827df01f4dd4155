"""Golden fixture for tests/test_gpu_dropin.py: the reference's own IRSDE + ConditionalUNet on a CUDA device (TF32 off),
driven the way its deraining test.py and train.py drive them, with the seeded weights and inputs the tests use.

Needs a GPU (the noise comes from torch's CUDA generator, which the native sampler's torch-RNG mode reproduces) and the
reference staged under baseline/_ref (baseline/make_ref.py):
    python tests/golden/make_golden_dropin.py [OUT_DIR]        # writes OUT_DIR/reference_golden_dropin.pt
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "baseline")]

import ref_loader  # noqa: E402
from test_gpu_dropin import NET_ARGS, SDE_ARGS, SEED, images, to_tensor, weights  # noqa: E402


def reference_net(mods, dev):
    net = mods.ConditionalUNet(*NET_ARGS)
    net.load_state_dict(weights(), strict=True)
    return net.to(dev)


def test_py_outputs(util, mods, dev, mode):
    net = reference_net(mods, dev).eval()
    sde = util.IRSDE(device=dev, **SDE_ARGS)
    sde.set_model(net)
    torch.manual_seed(SEED)
    outs = []
    for gt, lq in images():
        LQ, GT = to_tensor(lq), to_tensor(gt)
        noisy = sde.noise_state(LQ)
        sde.set_mu(LQ.to(dev))
        with torch.no_grad():
            out = getattr(sde, "reverse_" + mode)(noisy.to(dev))
        outs.append(torch.from_numpy(util.tensor2img(out[0].float().cpu())))
        assert np.array_equal(util.tensor2img(LQ[0]), lq) and np.array_equal(util.tensor2img(GT[0]), gt)
    return outs


def training_outputs(util, mods, dev):
    ref_net = reference_net(mods, dev)
    wrapped = torch.nn.DataParallel(ref_net, device_ids=[0])
    sde = util.IRSDE(device=dev, **SDE_ARGS)
    sde.set_model(wrapped)
    g = torch.Generator().manual_seed(1)
    GT, LQ = torch.rand(2, 3, 24, 40, generator=g), torch.rand(2, 3, 24, 40, generator=g)
    torch.manual_seed(5)
    t, states = sde.generate_random_states(x0=GT, mu=LQ)
    opt = torch.optim.SGD(ref_net.parameters(), lr=1e-2)

    def validate():
        wrapped.eval()
        sde.set_mu(LQ.to(dev))
        torch.manual_seed(9)
        with torch.no_grad():
            out = sde.reverse_posterior(LQ.to(dev) + 0.03)
        wrapped.train()
        return out.cpu()

    a = validate()
    torch.manual_seed(11)
    ts, st = sde.generate_random_states(x0=GT, mu=LQ)
    loss = sde.noise_fn(st, ts.squeeze().to(dev)).pow(2).mean()
    loss.backward()
    opt.step()
    b = validate()
    return dict(t=t.cpu(), states=states.cpu(), a=a, b=b)


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    util, mods = ref_loader.load("deraining")
    gold = dict(test_py={m: test_py_outputs(util, mods, dev, m) for m in ("posterior", "sde")},
                training=training_outputs(util, mods, dev))
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "reference_golden_dropin.pt")
    torch.save(gold, path)
    print("wrote", path, os.path.getsize(path))


if __name__ == "__main__":
    main()
