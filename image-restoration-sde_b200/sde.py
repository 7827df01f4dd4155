"""``IRSDE`` / ``DenoisingSDE`` with the reference's public surface (codes/utils/sde_utils.py:80-361,
373-593) on top of the native sm_100a sampler.

Host logic kept in Python: the theta/sigma schedules (a few hundred floats, computed once with the same
torch ops as the reference so they are bit-identical) and the per-timestep scalar tables handed to the
fused update kernel.  Everything per-pixel (network forward, drift/diffusion update, the T-step loop)
runs in the CUDA library; there is no CPU or eager-PyTorch fallback for the sampler.
"""
import ctypes
import math
import os

import torch

from . import _lib
from .unet import ConditionalUNet


def _unwrap(model):
    # DataParallel / DistributedDataParallel hand us a wrapper (models/denoising_model.py:37-42,
    # test.py:71); the native sampler owns batching itself, so use the underlying module.
    m = getattr(model, "module", model)
    if m is None or isinstance(m, ConditionalUNet):
        return m
    # A foreign nn.Module with the reference ConditionalUNet's state-dict layout (e.g. the reference's own PyTorch class
    # being trained by autograd in train.py): sample through a native shadow that re-reads its parameters (unet.adopt).
    # Opt out with IRSDE_B200_ADOPT=0; modules in training mode are left alone (autograd needs the PyTorch forward).
    if isinstance(m, torch.nn.Module) and os.environ.get("IRSDE_B200_ADOPT", "1") != "0" and not m.training:
        sh = getattr(m, "_irsde_b200_shadow", None)
        if sh is None:
            from .unet import adopt
            sh = adopt(m) or False
            try:
                object.__setattr__(m, "_irsde_b200_shadow", sh)
            except Exception:
                pass
        if sh:
            return sh
    return m


class _SDEBase:
    _kind = "irsde"

    def _setup(self, max_sigma, T, schedule, eps, device):
        self.T = T
        self.device = device
        # schedules: same torch ops as sde_utils.py:91-144 / :384-417 (bit-identical tables)
        if schedule == "cosine":
            timesteps = T + 2
            x = torch.linspace(0, timesteps, timesteps + 1, dtype=torch.float32)
            ac = torch.cos(((x / timesteps) + 0.008) / (1 + 0.008) * math.pi * 0.5) ** 2
            ac = ac / ac[0]
            thetas = 1 - ac[1:-1]
        elif schedule == "linear" or self._kind == "dsde":
            timesteps = T + 1
            scale = 1000 / timesteps
            thetas = torch.linspace(scale * 0.0001, scale * 0.02, timesteps, dtype=torch.float32)
        elif schedule == "constant":
            thetas = torch.ones(T + 1, dtype=torch.float32)
        else:
            raise NotImplementedError("Not implemented such schedule yet!!! (%r)" % (schedule,))
        sigmas = torch.sqrt(max_sigma ** 2 * 2 * thetas)
        thetas_cumsum = torch.cumsum(thetas, dim=0) - thetas[0]
        self.dt = -1 / thetas_cumsum[-1] * math.log(eps)  # 0-dim CPU tensor, like the reference
        sigma_bars = torch.sqrt(max_sigma ** 2 * (1 - torch.exp(-2 * thetas_cumsum * self.dt)))
        self._cpu = dict(thetas=thetas, sigmas=sigmas, thetas_cumsum=thetas_cumsum, sigma_bars=sigma_bars)
        self.thetas = thetas.to(device)
        self.sigmas = sigmas.to(device)
        self.thetas_cumsum = thetas_cumsum.to(device)
        self.sigma_bars = sigma_bars.to(device)
        self.mu = 0.
        self.model = None
        self._step_ctx = None
        _SDEBase._next_uid = getattr(_SDEBase, "_next_uid", 0) + 1
        self._uid = _SDEBase._next_uid  # never reused, unlike id(): names this sampler as the owner of uploaded tables
        self._coeff_cache = {}
        self.use_graph = os.environ.get("IRSDE_B200_GRAPH", "1") != "0"
        self.rng = os.environ.get("IRSDE_B200_RNG", "torch")  # "torch": randn_like per step; "philox": in-kernel
        self.seed = 0
        self.seed_auto_increment = True   # a fresh Philox seed per chain; False: (seed, image uid, t) fully decide the noise
        self.image_base = 0               # uid of the first image of the next batch (Philox is keyed per image)
        self.image_uids = None            # or explicit uids, one per image of the next batch

    # ---- per-timestep scalars in the reference's op order (0-dim fp32 tensor math) ----------------
    def _coeff_table(self, mode):
        c = self._cpu
        th, sg, cs, sb, dt = c["thetas"], c["sigmas"], c["thetas_cumsum"], c["sigma_bars"], self.dt
        T = self.T
        tab = torch.zeros(T + 1, _lib.NUM_COEF, dtype=torch.float32)
        sqdt = math.sqrt(dt)
        for t in range(1, T + 1):
            if mode == _lib.MODE_SDE:
                row = [th[t], sg[t] ** 2, sb[t], dt, sg[t], sqdt]
            elif mode == _lib.MODE_ODE:
                row = [th[t], 0.5 * sg[t] ** 2, sb[t], dt]
            elif mode == _lib.MODE_POSTERIOR:
                A0 = torch.exp(cs[t] * dt)
                A = torch.exp(-th[t] * dt)
                B = torch.exp(-cs[t] * dt)
                C = torch.exp(-cs[t - 1] * dt)
                term1 = A * (1 - C ** 2) / (1 - B ** 2)
                term2 = C * (1 - A ** 2) / (1 - B ** 2)
                A2 = torch.exp(-2 * th[t] * dt)
                B2 = torch.exp(-2 * cs[t] * dt)
                C2 = torch.exp(-2 * cs[t - 1] * dt)
                var = (1 - A2) * (1 - C2) / (1 - B2)
                std = (0.5 * torch.log(torch.clamp(var, min=1e-20 * dt))).exp() * self.max_sigma
                row = [A0, sb[t], term1, term2, std]
            elif mode == _lib.MODE_DSDE_SDE:
                A = torch.exp(-2 * cs[t] * dt)
                row = [-0.5 * sg[t] ** 2 * (1 + A), sb[t], dt, sg[t], sqdt]
            else:
                A = torch.exp(-2 * cs[t] * dt)
                row = [-0.5 * sg[t] ** 2 * A, sb[t], dt]
            for k, v in enumerate(row):
                tab[t, k] = float(v)
        return tab

    def _upload_schedule(self, ctx):
        # The tables live in the native context, which belongs to the MODEL: two samplers sharing one network
        # (IRSDE(T=100) and IRSDE(T=50), different max_sigma / eps ...) would otherwise run on each other's
        # thetas / sigma_bars / coefficients.  Ownership is recorded on the context object itself (not by id(): ids
        # are reused after a context is closed) and the tables are re-uploaded whenever another sampler wrote last.
        sig = (self._uid, self.T, float(self.max_sigma), float(self.dt))
        if getattr(ctx, "_sched_sig", None) == sig:
            return
        c = self._cpu
        fa = lambda t: _lib.float_array(t.tolist())
        _lib.check(ctx.L.irsde_set_schedule(ctx.h, fa(c["thetas"]), fa(c["sigmas"]), fa(c["thetas_cumsum"]),
                                            fa(c["sigma_bars"]), float(self.dt), float(self.max_sigma), self.T), ctx.h)
        for mode in self._modes:
            if mode not in self._coeff_cache:
                self._coeff_cache[mode] = self._coeff_table(mode).reshape(-1).tolist()
            tab = torch.tensor(self._coeff_cache[mode])
            _lib.check(ctx.L.irsde_set_coeffs(ctx.h, mode, _lib.float_array(tab.tolist()), self.T), ctx.h)
        ctx._sched_sig = sig

    def _ctx_for(self, x):
        """Native context used for the update kernel: the model's if it is ours, else a private one."""
        if not x.is_cuda:
            raise RuntimeError("irsde_b200 samplers run on CUDA (sm_100a) only; there is no CPU path")
        m = _unwrap(self.model) if self.model is not None else None
        if isinstance(m, ConditionalUNet):
            ctx = m.sync_weights(x.device)
        else:
            idx = x.device.index if x.device.index is not None else torch.cuda.current_device()
            if self._step_ctx is None or self._step_ctx[0] != idx:
                self._step_ctx = (idx, _lib.Context(3, 3, 4, 1, _lib.NET_CONDITIONAL if self._kind == "irsde"
                                                    else _lib.NET_DENOISING, _lib.PREC_FP32, idx))
            ctx = self._step_ctx[1]
        self._upload_schedule(ctx)
        return ctx

    def _apply_image_ids(self, ctx, B, st):
        if self.image_uids is not None:
            u = [int(v) for v in self.image_uids]
            if len(u) != B:
                raise ValueError("image_uids must hold one uid per image of the batch")
            arr = (ctypes.c_uint64 * B)(*u)
            _lib.check(ctx.L.irsde_set_image_uids(ctx.h, arr, B, ctypes.c_void_p(st)), ctx.h)
        else:
            _lib.check(ctx.L.irsde_set_image_base(ctx.h, int(self.image_base)), ctx.h)

    def _native_step(self, mode, x, mu, noise, z, t):
        ctx = self._ctx_for(x)
        x = x.contiguous().float()
        noise = noise.contiguous().float()
        out = torch.empty_like(x)
        p = lambda a: ctypes.c_void_p(a.data_ptr()) if a is not None else None
        if mu is not None:  # IRSDE starts with mu = 0. (a Python float, like the reference): broadcast it
            mu = torch.as_tensor(mu, dtype=torch.float32, device=x.device).expand_as(x).contiguous()
        if z is not None:
            z = z.contiguous().float()
        with torch.cuda.device(x.device):
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(ctx.L.irsde_step(ctx.h, mode, p(x), p(mu), p(noise), p(z), int(t), p(out), x.numel(),
                                        ctypes.c_void_p(st)), ctx.h)
        return out

    def _native_chain(self, mode, xt, mu, T, zs=None, lens_info=None):
        """Whole loop in the library: T network forwards + T fused updates (one captured step graph).  ``lens_info``: the
        lens network's camera rows, set once for the chain (they do not depend on t)."""
        m = _unwrap(self.model)
        ctx = self._ctx_for(xt)
        if lens_info is not None:
            m.set_lens(lens_info, xt.device)
        x = xt.contiguous().float()
        B, C, H, W = x.shape
        if mu is not None:
            mu = torch.as_tensor(mu, dtype=torch.float32, device=x.device).expand_as(x).contiguous()
        need_z = mode in (_lib.MODE_SDE, _lib.MODE_POSTERIOR, _lib.MODE_DSDE_SDE)
        if need_z and zs is None and self.rng == "torch":
            # same generator calls as the reference: one randn_like(x) per step in loop order
            zs = torch.stack([torch.randn_like(x) for _ in range(T)]) if T > 0 else None
        if zs is not None:
            zs = zs.contiguous().float()
            if zs.shape[0] < T or zs[0].numel() != x.numel():
                raise ValueError("zs must be [>=T, B, C, H, W]")
        out = torch.empty_like(x)
        p = lambda a: ctypes.c_void_p(a.data_ptr()) if a is not None else None
        with torch.cuda.device(x.device):
            st = torch.cuda.current_stream().cuda_stream
            self._apply_image_ids(ctx, B, st)
            _lib.check(ctx.L.irsde_reverse(ctx.h, mode, p(x), p(mu), p(zs), p(out), B, H, W, int(T), int(self.seed),
                                           1 if self.use_graph else 0, ctypes.c_void_p(st)), ctx.h)
        if self.seed_auto_increment:
            self.seed += 1
        self._keep = (x, mu, zs)  # keep inputs alive until the stream consumed them
        return out

    def _fast(self, kwargs, save_states):
        m = _unwrap(self.model) if self.model is not None else None
        if not isinstance(m, ConditionalUNet) or save_states:
            return False
        if getattr(m, "lens", False):  # the lens network's one keyword: set once per chain; without it the loop raises KeyError
            return set(kwargs) == {"lens_info"}
        return not kwargs

    @staticmethod
    def _save(x, t, T_total, save_dir):
        import torchvision.utils as tvutils
        interval = T_total // 100  # ZeroDivisionError for T<100, exactly like sde_utils.py:260-261
        if t % interval == 0:
            idx = t // interval
            os.makedirs(save_dir, exist_ok=True)
            tvutils.save_image(x.data, f"{save_dir}/state_{idx}.png", normalize=False)


class IRSDE(_SDEBase):
    """Mean-reverting SDE sampler; same constructor/attributes/methods as sde_utils.py:80-361."""
    _kind = "irsde"
    _modes = (_lib.MODE_SDE, _lib.MODE_ODE, _lib.MODE_POSTERIOR)

    def __init__(self, max_sigma, T=100, schedule="cosine", eps=0.01, device=None):
        self.max_sigma = max_sigma / 255 if max_sigma >= 1 else max_sigma
        self._setup(self.max_sigma, T, schedule, eps, device)

    # -- reference surface ---------------------------------------------------------------------------
    def set_mu(self, mu):
        self.mu = mu

    def set_model(self, model):
        self.model = model

    def mu_bar(self, x0, t):
        return self.mu + (x0 - self.mu) * torch.exp(-self.thetas_cumsum[t] * self.dt)

    def sigma_bar(self, t):
        return self.sigma_bars[t]

    def sigma(self, t):
        return self.sigmas[t]

    def theta(self, t):
        return self.thetas[t]

    def get_score_from_noise(self, noise, t):
        return -noise / self.sigma_bar(t)

    def score_fn(self, x, t, **kwargs):
        noise = self.model(x, self.mu, t, **kwargs)
        return self.get_score_from_noise(noise, t)

    def noise_fn(self, x, t, **kwargs):
        return self.model(x, self.mu, t, **kwargs)

    def get_real_noise(self, xt, x0, t):
        return (xt - self.mu_bar(x0, t)) / self.sigma_bar(t)

    def get_real_score(self, xt, x0, t):
        return -(xt - self.mu_bar(x0, t)) / self.sigma_bar(t) ** 2

    def get_init_state_from_noise(self, xt, noise, t):
        A = torch.exp(self.thetas_cumsum[t] * self.dt)
        return (xt - self.mu - self.sigma_bar(t) * noise) * A + self.mu

    # single steps -> fused CUDA kernel (noise-parameterised; score = -noise/sigma_bar inside)
    def reverse_sde_step(self, x, score, t):
        noise = -score * self.sigma_bar(t)
        return self._native_step(_lib.MODE_SDE, x, self.mu, noise, torch.randn_like(x), t)

    def reverse_ode_step(self, x, score, t):
        noise = -score * self.sigma_bar(t)
        return self._native_step(_lib.MODE_ODE, x, self.mu, noise, None, t)

    def reverse_posterior_step(self, xt, noise, t):
        return self._native_step(_lib.MODE_POSTERIOR, xt, self.mu, noise, torch.randn_like(xt), t)

    def _loop(self, mode, name, xt, T, save_states, save_dir, kwargs, zs=None):
        T = self.T if T < 0 else T
        if self._fast(kwargs, save_states):
            return self._native_chain(mode, xt, self.mu, T, zs, kwargs.get("lens_info"))
        x = xt.clone()
        for i, t in enumerate(reversed(range(1, T + 1))):
            noise = self.noise_fn(x, t, **kwargs)
            need_z = mode != _lib.MODE_ODE
            z = (zs[i] if zs is not None else torch.randn_like(x)) if need_z else None
            x = self._native_step(mode, x, self.mu, noise, z, t)
            if save_states:
                self._save(x, t, self.T, save_dir)
        return x

    def reverse_sde(self, xt, T=-1, save_states=False, save_dir="sde_state", zs=None, **kwargs):
        return self._loop(_lib.MODE_SDE, "sde", xt, T, save_states, save_dir, kwargs, zs)

    def reverse_ode(self, xt, T=-1, save_states=False, save_dir="ode_state", zs=None, **kwargs):
        return self._loop(_lib.MODE_ODE, "ode", xt, T, save_states, save_dir, kwargs, zs)

    def reverse_posterior(self, xt, T=-1, save_states=False, save_dir="posterior_state", zs=None, **kwargs):
        return self._loop(_lib.MODE_POSTERIOR, "posterior", xt, T, save_states, save_dir, kwargs, zs)

    # training-time helpers (not on the sampling hot path; plain tensor algebra like the reference)
    def reverse_optimum_step(self, xt, x0, t):
        A = torch.exp(-self.thetas[t] * self.dt)
        B = torch.exp(-self.thetas_cumsum[t] * self.dt)
        C = torch.exp(-self.thetas_cumsum[t - 1] * self.dt)
        term1 = A * (1 - C ** 2) / (1 - B ** 2)
        term2 = C * (1 - A ** 2) / (1 - B ** 2)
        return term1 * (xt - self.mu) + term2 * (x0 - self.mu) + self.mu

    def reverse_sde_step_mean(self, x, score, t):
        return x - (self.thetas[t] * (self.mu - x) - self.sigmas[t] ** 2 * score) * self.dt

    # forward-process / diagnostic helpers of the reference (sde_utils.py:39-52,170-182,207-217,240-251,326-333); not on the
    # sampling hot path, plain tensor algebra on whatever device the inputs live on
    def drift(self, x, t):
        return self.thetas[t] * (self.mu - x) * self.dt

    def dispersion(self, x, t):
        return self.sigmas[t] * (torch.randn_like(x) * math.sqrt(self.dt)).to(self.device)

    def sde_reverse_drift(self, x, score, t):
        return (self.thetas[t] * (self.mu - x) - self.sigmas[t] ** 2 * score) * self.dt

    def ode_reverse_drift(self, x, score, t):
        return (self.thetas[t] * (self.mu - x) - 0.5 * self.sigmas[t] ** 2 * score) * self.dt

    def forward_step(self, x, t):
        return x + self.drift(x, t) + self.dispersion(x, t)

    def forward(self, x0, T=-1, save_dir=None):
        """x(0) -> x(T) by Euler-Maruyama steps of the forward SDE (the reference also dumps every state as a PNG into
        ``save_dir='forward_state'``; here only when a directory is given)."""
        T = self.T if T < 0 else T
        x = x0.clone()
        for t in range(1, T + 1):
            x = self.forward_step(x, t)
            if save_dir:
                import torchvision.utils as tvutils
                os.makedirs(save_dir, exist_ok=True)
                tvutils.save_image(x.data, f"{save_dir}/state_{t}.png", normalize=False)
        return x

    def reverse_optimum_std(self, t):
        A = torch.exp(-2 * self.thetas[t] * self.dt)
        B = torch.exp(-2 * self.thetas_cumsum[t] * self.dt)
        C = torch.exp(-2 * self.thetas_cumsum[t - 1] * self.dt)
        var = (1 - A) * (1 - C) / (1 - B)
        floor = (1e-20 * self.dt).to(self.device)
        return (0.5 * torch.log(torch.clamp(var, min=floor))).exp() * self.max_sigma

    def optimal_reverse(self, xt, x0, T=-1):
        T = self.T if T < 0 else T
        x = xt.clone()
        for t in reversed(range(1, T + 1)):
            x = self.reverse_optimum_step(x, x0, t)
        return x

    def weights(self, t):
        return torch.exp(-self.thetas_cumsum[t] * self.dt)

    def generate_random_states(self, x0, mu):
        """Training-time state sampler (sde_utils.py:343-358; train.py:236).  Same generator calls as the reference
        (one CPU randint for the timesteps, one randn_like on the device); on a CUDA device the mean-reversion + noising is
        ONE fused kernel (irsde_random_states) that reproduces the torch expression bit for bit."""
        x0 = x0.to(self.device)
        mu = mu.to(self.device)
        self.set_mu(mu)
        batch = x0.shape[0]
        timesteps = torch.randint(1, self.T + 1, (batch, 1, 1, 1)).long()
        if not (x0.is_cuda and x0.dtype == torch.float32 and mu.shape == x0.shape):
            state_mean = self.mu_bar(x0, timesteps)
            noises = torch.randn_like(state_mean)
            noise_level = self.sigma_bar(timesteps)
            noisy_states = noises * noise_level + state_mean
            return timesteps, noisy_states.to(torch.float32)
        noises = torch.randn_like(x0)
        t = timesteps.reshape(-1).to(x0.device)
        w = torch.exp(-self.thetas_cumsum[t] * self.dt).float().contiguous()     # the reference's per-image scalars, same ops
        sb = self.sigma_bars[t].float().contiguous()
        x0c, muc = x0.contiguous(), mu.contiguous()
        out = torch.empty_like(x0c)
        p = lambda a: ctypes.c_void_p(a.data_ptr())
        with torch.cuda.device(x0.device):
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(_lib.load().irsde_random_states(p(x0c), p(muc), p(noises), p(w), p(sb), p(out), batch, x0c[0].numel(),
                                                       ctypes.c_void_p(st)))
        return timesteps, out

    def noise_state(self, tensor):
        # called on CPU tensors by test.py:104 before feed_data: plain torch, like the reference
        if not (tensor.is_cuda and self.rng == "philox"):
            return tensor + torch.randn_like(tensor) * self.max_sigma
        # device path (SURVEY 8 f-2): x_T drawn by the library's per-image Philox, nothing crosses PCIe
        ctx = self._ctx_for(tensor)
        mu = tensor.contiguous().float()
        out = torch.empty_like(mu)
        B = mu.shape[0] if mu.dim() == 4 else 1
        with torch.cuda.device(mu.device):
            st = torch.cuda.current_stream().cuda_stream
            self._apply_image_ids(ctx, B, st)
            _lib.check(ctx.L.irsde_noise_state_images(ctx.h, ctypes.c_void_p(mu.data_ptr()), ctypes.c_void_p(out.data_ptr()), B,
                                                      mu.numel() // B, int(self.seed), ctypes.c_void_p(st)), ctx.h)
        return out


class DenoisingSDE(_SDEBase):
    """Denoising SDE sampler (sde_utils.py:373-593): no mean reversion, model(x, t) without condition."""
    _kind = "dsde"
    _modes = (_lib.MODE_DSDE_SDE, _lib.MODE_DSDE_ODE)

    def __init__(self, max_sigma, T, schedule="cosine", device=None):
        self.max_sigma = max_sigma / 255 if max_sigma > 1 else max_sigma
        self._setup(self.max_sigma, T, schedule, 0.04, device)

    def set_model(self, model):
        self.model = model

    def sigma(self, t):
        return self.sigmas[t]

    def theta(self, t):
        return self.thetas[t]

    def mu_bar(self, x0, t):
        return x0

    def sigma_bar(self, t):
        return self.sigma_bars[t]

    def get_score_from_noise(self, noise, t):
        return -noise / self.sigma_bar(t)

    def get_init_state_from_noise(self, x, noise, t):
        return x - self.sigma_bar(t) * noise

    def get_init_state_from_score(self, x, score, t):
        return x + self.sigma_bar(t) ** 2 * score

    def score_fn(self, x, t):
        noise = self.model(x, t)
        return self.get_score_from_noise(noise, t)

    def get_real_noise(self, xt, x0, t):
        return (xt - self.mu_bar(x0, t)) / self.sigma_bar(t)

    def get_real_score(self, xt, x0, t):
        return -(xt - self.mu_bar(x0, t)) / self.sigma_bar(t) ** 2

    def reverse_sde_step(self, x, score, t):
        return self._native_step(_lib.MODE_DSDE_SDE, x, None, -score * self.sigma_bar(t), torch.randn_like(x), t)

    def reverse_ode_step(self, x, score, t):
        return self._native_step(_lib.MODE_DSDE_ODE, x, None, -score * self.sigma_bar(t), None, t)

    def _loop(self, mode, xt, x0, T, save_states, save_dir, zs=None):
        if torch.is_tensor(T):  # denoising_model.py:163 passes a 0-dim LongTensor
            T = int(T)
        T = self.T if T < 0 else T
        if x0 is None and self._fast({}, save_states):
            return self._native_chain(mode, xt, None, T, zs)
        x = xt.clone()
        for i, t in enumerate(reversed(range(1, T + 1))):
            if x0 is not None and mode == _lib.MODE_DSDE_SDE:
                noise = self.get_real_noise(x, x0, t)
            else:
                noise = self.model(x, t)
            z = (zs[i] if zs is not None else torch.randn_like(x)) if mode == _lib.MODE_DSDE_SDE else None
            x = self._native_step(mode, x, None, noise, z, t)
            if save_states:
                self._save(x, t, self.T, save_dir)
        return x

    def reverse_sde(self, xt, x0=None, T=-1, save_states=False, save_dir="sde_state", zs=None):
        return self._loop(_lib.MODE_DSDE_SDE, xt, x0, T, save_states, save_dir, zs)

    def reverse_ode(self, xt, x0=None, T=-1, save_states=False, save_dir="ode_state", zs=None):
        return self._loop(_lib.MODE_DSDE_ODE, xt, x0, T, save_states, save_dir, zs)

    # reference helpers off the sampling path (sde_utils.py:446-459,556-571): plain tensor algebra
    def drift(self, x, x0, t):
        return self.thetas[t] * (x0 - x) * self.dt

    def sde_reverse_drift(self, x, score, t):
        A = torch.exp(-2 * self.thetas_cumsum[t] * self.dt)
        return -0.5 * self.sigmas[t] ** 2 * (1 + A) * score * self.dt

    def ode_reverse_drift(self, x, score, t):
        A = torch.exp(-2 * self.thetas_cumsum[t] * self.dt)
        return -0.5 * self.sigmas[t] ** 2 * A * score * self.dt

    def dispersion(self, x, t):
        return self.sigmas[t] * (torch.randn_like(x) * math.sqrt(self.dt)).to(self.device)

    def reverse_sde_step_mean(self, x, score, t):
        return x - self.sde_reverse_drift(x, score, t)

    def optimal_reverse(self, xt, x0, T=-1):
        T = self.T if T < 0 else T
        x = xt.clone()
        for t in reversed(range(1, T + 1)):
            x = self.reverse_optimum_step(x, x0, t)
        return x

    def get_optimal_timestep(self, sigma, eps=1e-6):
        sigma = sigma / 255 if sigma > 1 else sigma
        thetas_cumsum_hat = -1 / (2 * self.dt) * math.log(1 - sigma ** 2 / self.max_sigma ** 2 + eps)
        T = torch.argmin((self.thetas_cumsum - thetas_cumsum_hat).abs())
        return T

    def reverse_optimum_step(self, xt, x0, t):
        A = torch.exp(-self.thetas[t] * self.dt)
        B = torch.exp(-self.thetas_cumsum[t] * self.dt)
        C = torch.exp(-self.thetas_cumsum[t - 1] * self.dt)
        term1 = A * (1 - C ** 2) / (1 - B ** 2)
        term2 = C * (1 - A ** 2) / (1 - B ** 2)
        return term1 * (xt - x0) + term2 * (x0 - x0) + x0

    def weights(self, t):
        return self.sigmas[t] ** 2

    def generate_random_states(self, x0):
        x0 = x0.to(self.device)
        batch = x0.shape[0]
        timesteps = torch.randint(1, self.T + 1, (batch, 1, 1, 1)).long()
        noises = torch.randn_like(x0, dtype=torch.float32)
        noise_level = self.sigma_bar(timesteps)
        noisy_states = noises * noise_level + x0
        return timesteps, noisy_states
