"""Restatement of the k-diffusion 0.1.1 pieces the reference calls.

TEST INFRASTRUCTURE (see oracle/__init__.py).

PARITY UNPINNED: ``k-diffusion==0.1.1`` (reference ``setup.py:21``) is an
un-vendored third-party dependency that is absent from ``/root/reference`` and
from this image, and so is ``torchsde`` (its Brownian-tree noise source).  The
formulas below restate the published algorithms (Karras et al. 2022 for the
v-objective preconditioning; Lu et al. 2022 DPM-Solver++ multistep SDE
variants as implemented in k-diffusion's ``sampling.py``) and are anchored on
the reference's call sites:

* ``K.external.VDenoiser(model_fn)``               inference/sampling.py:159,252
* ``K.sampling.get_sigmas_polyexponential(...)``   inference/sampling.py:165
* ``K.sampling.sample_dpmpp_2m_sde(...)``          inference/sampling.py:225-226
* ``K.sampling.sample_dpmpp_3m_sde(...)``          inference/sampling.py:227-228
* ``K.utils.append_dims``                          inference/sampling.py:133

Noise: k-diffusion draws the SDE noise from a torchsde Brownian tree.  Its
increments over the disjoint ``[sigma_{i+1}, sigma_i]`` intervals, normalised
by sqrt(|t1-t0|), are i.i.d. N(0, 1), so the default here is one
``torch.randn_like`` per step; parity runs inject an explicit
``noise_sampler(sigma, sigma_next)`` into both loops.
"""
import math

import torch


def append_dims(x, target_dims):
    """Right-pad ``x`` with singleton dims up to ``target_dims`` dimensions."""
    extra = target_dims - x.ndim
    if extra < 0:
        raise ValueError("input has more dims than the target")
    return x[(...,) + (None,) * extra]


def get_sigmas_polyexponential(n, sigma_min, sigma_max, rho=1.0, device="cpu"):
    """n noise levels, polynomial in log-sigma, followed by a terminal 0."""
    ramp = torch.linspace(1, 0, n, device=device) ** rho
    log_lo, log_hi = math.log(sigma_min), math.log(sigma_max)
    sigmas = torch.exp(ramp * (log_hi - log_lo) + log_lo)
    return torch.cat([sigmas, sigmas.new_zeros([1])])


class VDenoiser(torch.nn.Module):
    """v-objective preconditioning with sigma_data = 1.

    D(x, sigma) = F(x * c_in, t(sigma)) * c_out + x * c_skip,
    c_skip = 1/(sigma^2+1), c_out = -sigma/sqrt(sigma^2+1),
    c_in = 1/sqrt(sigma^2+1), t = atan(sigma) * 2/pi.
    """

    sigma_data = 1.0

    def __init__(self, inner_model):
        super().__init__()
        self.inner_model = inner_model

    def get_scalings(self, sigma):
        sd2 = self.sigma_data ** 2
        denom = sigma ** 2 + sd2
        c_skip = sd2 / denom
        c_out = -sigma * self.sigma_data / denom ** 0.5
        c_in = 1 / denom ** 0.5
        return c_skip, c_out, c_in

    @staticmethod
    def sigma_to_t(sigma):
        return sigma.atan() / math.pi * 2

    def forward(self, input, sigma, **kwargs):
        c_skip, c_out, c_in = (append_dims(c, input.ndim) for c in self.get_scalings(sigma))
        v = self.inner_model(input * c_in, self.sigma_to_t(sigma), **kwargs)
        return v * c_out + input * c_skip


def default_noise_sampler(x):
    return lambda sigma, sigma_next: torch.randn_like(x)


@torch.no_grad()
def sample_dpmpp_2m_sde(model, x, sigmas, extra_args=None, callback=None, disable=None,
                        eta=1.0, s_noise=1.0, noise_sampler=None, solver_type="midpoint"):
    """DPM-Solver++(2M) SDE; one model call per step."""
    if solver_type not in ("heun", "midpoint"):
        raise ValueError("solver_type must be 'heun' or 'midpoint'")
    noise_sampler = default_noise_sampler(x) if noise_sampler is None else noise_sampler
    extra_args = {} if extra_args is None else extra_args
    ones = x.new_ones([x.shape[0]])
    prev_den, prev_h = None, None
    for i in range(len(sigmas) - 1):
        den = model(x, sigmas[i] * ones, **extra_args)
        if callback is not None:
            callback({"x": x, "i": i, "sigma": sigmas[i], "sigma_hat": sigmas[i], "denoised": den})
        if sigmas[i + 1] == 0:
            x = den
            h = None
        else:
            lam_cur, lam_next = -sigmas[i].log(), -sigmas[i + 1].log()
            h = lam_next - lam_cur
            eta_h = eta * h
            x = sigmas[i + 1] / sigmas[i] * (-eta_h).exp() * x + (-h - eta_h).expm1().neg() * den
            if prev_den is not None:
                r = prev_h / h
                if solver_type == "heun":
                    x = x + ((-h - eta_h).expm1().neg() / (-h - eta_h) + 1) * (1 / r) * (den - prev_den)
                else:
                    x = x + 0.5 * (-h - eta_h).expm1().neg() * (1 / r) * (den - prev_den)
            if eta:
                x = x + noise_sampler(sigmas[i], sigmas[i + 1]) * sigmas[i + 1] \
                    * (-2 * eta_h).expm1().neg().sqrt() * s_noise
        prev_den, prev_h = den, h
    return x


@torch.no_grad()
def sample_dpmpp_3m_sde(model, x, sigmas, extra_args=None, callback=None, disable=None,
                        eta=1.0, s_noise=1.0, noise_sampler=None):
    """DPM-Solver++(3M) SDE; one model call per step."""
    noise_sampler = default_noise_sampler(x) if noise_sampler is None else noise_sampler
    extra_args = {} if extra_args is None else extra_args
    ones = x.new_ones([x.shape[0]])
    den_1 = den_2 = None
    h_1 = h_2 = None
    for i in range(len(sigmas) - 1):
        den = model(x, sigmas[i] * ones, **extra_args)
        if callback is not None:
            callback({"x": x, "i": i, "sigma": sigmas[i], "sigma_hat": sigmas[i], "denoised": den})
        if sigmas[i + 1] == 0:
            x = den
            h = None
        else:
            lam_cur, lam_next = -sigmas[i].log(), -sigmas[i + 1].log()
            h = lam_next - lam_cur
            h_eta = h * (eta + 1)
            x = torch.exp(-h_eta) * x + (-h_eta).expm1().neg() * den
            if h_2 is not None:
                r0, r1 = h_1 / h, h_2 / h
                d1_0 = (den - den_1) / r0
                d1_1 = (den_1 - den_2) / r1
                d1 = d1_0 + (d1_0 - d1_1) * r0 / (r0 + r1)
                d2 = (d1_0 - d1_1) / (r0 + r1)
                phi_2 = h_eta.neg().expm1() / h_eta + 1
                phi_3 = phi_2 / h_eta - 0.5
                x = x + phi_2 * d1 - phi_3 * d2
            elif h_1 is not None:
                r = h_1 / h
                d = (den - den_1) / r
                phi_2 = h_eta.neg().expm1() / h_eta + 1
                x = x + phi_2 * d
            if eta:
                x = x + noise_sampler(sigmas[i], sigmas[i + 1]) * sigmas[i + 1] \
                    * (-2 * h * eta).expm1().neg().sqrt() * s_noise
        den_1, den_2 = den, den_1
        h_1, h_2 = h, h_1
    return x


# ---------------------------------------------------------------------------------------------
# The reference's own sampler front end and inpainting mask (these ARE part of the reference and are pinned
# against its outputs by tests/test_oracle_vs_reference.py).
# ---------------------------------------------------------------------------------------------
def get_bmask(i, steps, mask):
    """inference/sampling.py:120-124: hard mask that shrinks as the step index grows."""
    return torch.where(mask <= (i + 1) / steps, 1, 0)


def build_mask(sample_size, mask_args):
    """inference/generation.py:270-292: soft keep-mask over the latent positions (1 = keep the init audio),
    Hann ramps of softnessL / softnessR percent on the two edges, scaled down by `marination`."""
    pct = lambda key: mask_args[key] / 100.0 * sample_size
    start, end = math.floor(pct("maskstart")), math.ceil(pct("maskend"))
    n_l, n_r = round(pct("softnessL")), round(pct("softnessR"))
    m = torch.zeros(sample_size)
    m[start:end] = 1
    m[start:start + n_l] = torch.hann_window(2 * n_l, periodic=False)[:n_l]
    m[end - n_r:end] = torch.hann_window(2 * n_r, periodic=False)[n_r:]
    if mask_args["marination"] > 0:
        m = m * (1 - mask_args["marination"])
    return m


def cut_paste(init, sample_size, mask_args):
    """inference/generation.py:197-210: move init[crop_from : crop_from + n] to paste_from (zeros elsewhere)."""
    crop_from = math.floor(mask_args["cropfrom"] / 100.0 * sample_size)
    paste_from = math.floor(mask_args["pastefrom"] / 100.0 * sample_size)
    paste_to = math.ceil(mask_args["pasteto"] / 100.0 * sample_size)
    n = min(paste_to - paste_from, sample_size - crop_from)
    out = init.new_zeros(init.shape)
    out[:, :, paste_from:paste_from + n] = init[:, :, crop_from:crop_from + n]
    return out


@torch.no_grad()
def sample_k(model_fn, noise, init_data=None, mask=None, steps=100, sampler_type="dpmpp-2m-sde", sigma_min=0.5,
             sigma_max=50, rho=1.0, noise_sampler=None, **extra_args):
    """inference/sampling.py:144-228 for the two multistep SDE samplers: sigma schedule (:165), initial noise
    scaled by sigma_0 (:167), variation start (:171-174), inpainting start + per-step callback that re-noises the
    kept region with this step's sigma and the shrinking hard mask (:175-199), plain sampling (:203-206).
    `noise_sampler` (not a reference argument) injects the SDE noise; None = randn_like like k-diffusion's default."""
    den = VDenoiser(model_fn)
    sigmas = get_sigmas_polyexponential(steps, sigma_min, sigma_max, rho)
    noise = noise * sigmas[0]
    callback = None
    if init_data is not None and mask is None:
        x = init_data + noise
    elif init_data is not None:
        b0 = get_bmask(0, steps, mask)
        x = (init_data + noise) * b0 + noise * (1 - b0)

        def callback(args):
            renoised = init_data + torch.randn_like(init_data) * args["sigma"]
            b = get_bmask(args["i"], steps, mask)
            args["x"][:, :, :] = renoised * b + args["x"] * (1 - b)
    else:
        x = noise
    fn = {"dpmpp-2m-sde": sample_dpmpp_2m_sde, "dpmpp-3m-sde": sample_dpmpp_3m_sde}[sampler_type]
    return fn(den, x, sigmas, extra_args=extra_args, callback=callback, noise_sampler=noise_sampler)
