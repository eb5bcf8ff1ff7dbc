"""Host-side diffusion schedules, bit-replicating the reference's fp32 coefficient arithmetic.

The reference rebuilds these tables with (mixed numpy/torch) fp32 tensor ops on every call
(ddim.py:25-55, util.py:46-75; ddpm_ddim_wrapper.py:194-199, 264-303); the per-step kernels in libcdx take
the resulting fp32 scalars as arguments, so the tables must be produced with exactly the same sequence of
IEEE fp32 operations.  We therefore evaluate the very same expressions with torch CPU tensors of shape [1]
(PyTorch here is host-side plumbing; nothing in this file touches the GPU).
"""
import numpy as np
import torch

from ._cabi import DdimCoef, PixelCoef


# ------------------------------------------------------------------------------------------ latent models
def ldm_alphas_cumprod(n_timestep=1000, linear_start=0.00085, linear_end=0.012):
    """make_beta_schedule('linear') (util.py:21-26) -> fp64 cumprod -> fp32 buffer (ddpm.py:117-138)."""
    betas = (torch.linspace(linear_start ** 0.5, linear_end ** 0.5, n_timestep, dtype=torch.float64) ** 2).numpy()
    return torch.tensor(np.cumprod(1.0 - betas, axis=0), dtype=torch.float32)


class DDIMSchedule:
    """DDIMSampler.make_schedule for (S, eta) plus the loop geometry of _ddpm_ddim_encoding / ddim_sampling_with_eps."""

    def __init__(self, S, eta, skip_steps=0, alphas_cumprod=None, num_ddpm_timesteps=1000):
        ac = ldm_alphas_cumprod(num_ddpm_timesteps) if alphas_cumprod is None else alphas_cumprod.to(torch.float32).cpu()
        assert ac.shape[0] == num_ddpm_timesteps, 'alphas have to be defined for each timestep'   # ddim.py:29
        c = num_ddpm_timesteps // S
        self.timesteps = np.asarray(list(range(0, num_ddpm_timesteps, c)))[:S] + 1            # util.py:46-61
        alphas = ac[self.timesteps]                                                          # fp32 torch
        alphas_prev = np.asarray([ac[0]] + ac[self.timesteps[:-1]].tolist())                 # fp64 numpy, util.py:67
        with np.errstate(all='ignore'):
            sigmas = eta * np.sqrt((1 - alphas_prev) / (1 - alphas) * (1 - alphas / alphas_prev))   # fp64 torch, util.py:70
            sqrt_1m = np.sqrt(1.0 - alphas)                                                      # fp32 torch, ddim.py:50
        self.total_steps = int(self.timesteps.shape[0])
        self.refine_steps = self.total_steps - skip_steps
        assert self.refine_steps >= 1
        self.eta = eta
        # loop order: iteration i uses index = refine_steps - 1 - i and timestep flip(timesteps)[-refine_steps:][i]
        time_range = np.flip(self.timesteps)[-self.refine_steps:]
        self.t_loop = [float(int(t)) for t in time_range]
        self.coef = []
        for i in range(self.refine_steps):
            index = self.refine_steps - 1 - i
            a_t = torch.full((1,), alphas[index])                      # ddim.py:570-573 (torch.full -> fp32)
            a_prev = torch.full((1,), alphas_prev[index])
            sigma_t = torch.full((1,), sigmas[index])
            s1m = torch.full((1,), sqrt_1m[index])
            self.coef.append(DdimCoef(
                sqrt_at=a_t.sqrt().item(),
                sqrt_1m_at=(1 - a_t).sqrt().item(),
                sqrt_1m_at_tab=s1m.item(),
                sqrt_aprev=a_prev.sqrt().item(),
                dir_coef=(1. - a_prev - sigma_t ** 2).sqrt().item(),
                sigma=sigma_t.item()))
        at = alphas[self.refine_steps - 1]                             # ddim.py:477-479
        self.sqrt_a_T = at.sqrt().item()
        self.sqrt_1ma_T = (1 - at).sqrt().item()

    def coef_array(self):
        return (DdimCoef * len(self.coef))(*self.coef)

    def t_array(self):
        import ctypes
        return (ctypes.c_float * len(self.t_loop))(*self.t_loop)


# ------------------------------------------------------------------------------------------ pixel models
class PixelSchedule:
    """Per-step scalars of DDPMDDIMWrapper.encode / generate (ddpm_ddim_wrapper.py:392-523)."""

    def __init__(self, sample_type, custom_steps, es_steps, eta=None, t_0=None, beta_start=1e-4, beta_end=2e-2, T=1000, var_type='fixedsmall'):
        if sample_type == 'ddim':
            assert eta > 0                                              # DW:333-334
        elif sample_type == 'ddpm':
            assert eta is None                                          # DW:335-336
        else:
            raise ValueError()
        self.sample_type, self.eta = sample_type, eta
        t_0 = 999 if t_0 is None else t_0
        betas64 = np.linspace(beta_start, beta_end, T, dtype=np.float64)            # diffusion_utils.py:5-9
        self.b = torch.from_numpy(betas64).float()                                   # DW:350-352
        ac = np.cumprod(1.0 - betas64, axis=0)
        ac_prev = np.append(1.0, ac[:-1])
        post_var = betas64 * (1.0 - ac_prev) / (1.0 - ac)
        if var_type == 'fixedlarge':                                                  # DW:362-363 (Ho-et-al checkpoints may use it)
            self.logvar = np.log(np.append(post_var[1], betas64[1:]))
        else:
            assert var_type == 'fixedsmall'
            self.logvar = np.log(np.maximum(post_var, 1e-20))                         # DW:356-373 (fp64)
        if (t_0 + 1) % custom_steps == 0:                                             # DW:393-400
            seq_inv = range(0, t_0 + 1, (t_0 + 1) // custom_steps)
            assert len(seq_inv) == custom_steps
        else:
            seq_inv = np.linspace(0, 1, custom_steps) * t_0
        seq_inv = [int(s) for s in list(seq_inv)][:es_steps]
        seq_inv_next = ([-1] + list(seq_inv[:-1]))[:es_steps]
        self.pairs = list(zip(reversed(seq_inv), reversed(seq_inv_next)))             # loop order (noisiest first)
        self.es_steps = es_steps
        self.cumprod = (1.0 - self.b).cumprod(dim=0)                                  # fp32, DW:194 (re-done per step there)
        at = self._extract(self.cumprod, es_steps - 1)                                # DW:483-484: es_steps-1 used as a timestep
        self.sqrt_a_T = at.sqrt().item()
        self.sqrt_1ma_T = (1 - at).sqrt().item()
        self.coef = [self.step_coef(i, j, eta) for i, j in self.pairs]
        self.t_loop = [float(i) for i, _ in self.pairs]

    @staticmethod
    def _extract(a, t):
        return torch.gather(torch.as_tensor(a, dtype=torch.float), 0, torch.tensor([int(t)]))   # diffusion_utils.py:12-20

    def step_coef(self, t, t_next, eta):
        b = self.b
        bt = self._extract(b, t)
        at = self._extract(self.cumprod, t)
        at_next = torch.ones_like(at) if t_next == -1 else self._extract(self.cumprod, t_next)   # DW:196-199
        c = PixelCoef()
        c.ddpm = 1 if self.sample_type == 'ddpm' else 0
        c.sqrt_at = at.sqrt().item()
        c.sqrt_1m_at = (1 - at).sqrt().item()
        c.sqrt_at_next = at_next.sqrt().item()
        if self.sample_type == 'ddim':
            c1 = eta * ((1 - at / at_next) * (1 - at_next) / (1 - at)).sqrt()                    # DW:217 / 273 / 300
            c2 = ((1 - at_next) - c1 ** 2).sqrt()
            c.c1, c.c2 = c1.item(), c2.item()
        else:
            c.w0 = (at_next.sqrt() * bt / (1 - at)).item()                                        # DW:291
            c.wt = ((1 - bt).sqrt() * (1 - at_next) / (1 - at)).item()                            # DW:292
            c.post_std = (bt * (1 - at_next) / (1 - at)).sqrt().item()                            # DW:295-297
            c.weight = (bt / torch.sqrt(1 - at)).item()                                           # DW:202
            c.inv_sqrt_1m_bt = (1 / torch.sqrt(1.0 - bt)).item()                                  # DW:204
            logvar = self._extract(self.logvar, t)
            c.std_model = torch.exp(0.5 * logvar).item()                                          # DW:208
            c.mask = 1.0 - float(t == 0)                                                          # DW:206
        return c

    def coef_array(self, coefs=None):
        coefs = self.coef if coefs is None else coefs
        return (PixelCoef * len(coefs))(*coefs)

    def same_as(self, other):
        """True when both schedules drive the samplers with the same numbers: sample type, eta, step pairs, betas, log-variances
        and every per-step scalar."""
        return (isinstance(other, PixelSchedule) and self.sample_type == other.sample_type and self.eta == other.eta
                and self.es_steps == other.es_steps and self.pairs == other.pairs and self.t_loop == other.t_loop
                and torch.equal(self.b, other.b) and np.array_equal(self.logvar, other.logvar)
                and (self.sqrt_a_T, self.sqrt_1ma_T) == (other.sqrt_a_T, other.sqrt_1ma_T)
                and bytes(self.coef_array()) == bytes(other.coef_array()))
