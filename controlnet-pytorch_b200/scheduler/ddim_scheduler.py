"""DDIM sampling (Song et al., "Denoising Diffusion Implicit Models", eq. 12) over a LinearNoiseScheduler's tables: a
strided schedule of S timesteps for the same eps-prediction models, with no retraining.  No counterpart in the
reference, whose tools walk the whole DDPM chain.

For step k of tau_0 > tau_1 > ... > tau_{S-1}, with a_t = alpha_cum_prod[tau_k] and a_p = alpha_cum_prod[tau_{k+1}]
(1.0 after the last step), the coefficient row is

    sigma_k = eta * sqrt((1 - a_p) / (1 - a_t)) * sqrt(1 - a_t / a_p)
    row_k   = [sqrt_one_minus_alpha_cum_prod[tau_k], sqrt_alpha_cum_prod[tau_k], sqrt(a_p),
               sqrt(max(1 - a_p - sigma_k^2, 0)), sigma_k, 1.0 if sigma_k > 0 else 0.0]

Columns 0, 1 and 2 are the base scheduler's fp32 values, so the x0 of a DDIM step is bit-identical to the DDPM step's;
columns 3 and 4 are evaluated in float64 from the fp32 alpha_cum_prod and rounded once.  The update itself is one fused
kernel (cnb_ddim_step).  eta = 0 is deterministic DDIM; eta = 1 with S = T is the DDPM posterior step.
"""
import math

import torch

from .. import ops
from .. import runtime as rt
from .schedule import StridedScheduler, step_inputs


class DDIMScheduler(StridedScheduler):
    """`base` is a LinearNoiseScheduler (DDPM or LDM betas).  The schedule is `timesteps` when given (strictly
    decreasing, inside [0, T)), otherwise `num_inference_steps` timesteps with the given spacing:
      "trailing": round(T - k T / S) - 1, k = 0 .. S-1 (round half to even), starting at T-1 where x_T ~ N(0, I);
      "leading":  (S-1-k) * (T // S), ending at 0.
    Attributes may be changed after construction; every call re-validates them."""
    TAG = "ddim"

    def __init__(self, base, num_inference_steps=50, eta=0.0, spacing="trailing", clip_sample=False, timesteps=None):
        self.eta = eta
        super().__init__(base, num_inference_steps, spacing, clip_sample, timesteps)

    def _params(self):
        eta = float(self.eta)
        if not (math.isfinite(eta) and eta >= 0.0):
            raise rt.CnbError(f"DDIMScheduler: eta must be a finite number >= 0 (got {self.eta!r})")
        return (eta,)

    def coef_table_host(self, steps=None):
        """fp32 [T, 6]: row tau_k is row_k of the module docstring; rows off the schedule are NaN, so that reading one
        by mistake poisons the output instead of passing unnoticed."""
        ts, (eta,), b = self.timesteps(steps), self._params(), self.base
        acp = b.alpha_cum_prod
        tab = torch.full((self.num_timesteps, 6), float("nan"), dtype=torch.float32)
        for k, t in enumerate(ts):
            last = k + 1 == len(ts)
            a_t = float(acp[t])
            a_p = 1.0 if last else float(acp[ts[k + 1]])
            sigma = eta * math.sqrt((1.0 - a_p) / (1.0 - a_t)) * math.sqrt(1.0 - a_t / a_p)
            tab[t, 0] = b.sqrt_one_minus_alpha_cum_prod[t]
            tab[t, 1] = b.sqrt_alpha_cum_prod[t]
            tab[t, 2] = 1.0 if last else b.sqrt_alpha_cum_prod[ts[k + 1]]
            tab[t, 3] = math.sqrt(max(1.0 - a_p - sigma * sigma, 0.0))
            tab[t, 4] = sigma
            tab[t, 5] = 1.0 if sigma > 0.0 else 0.0
        return tab

    def new_state(self, x):
        """DDIM carries nothing from one step to the next."""
        return {}

    def update(self, xt, eps, coef, **kw):
        """The fused update for one row of coef_table (ops.ddim_step and its keyword arguments)."""
        return ops.ddim_step(xt, eps, coef, clip_sample=bool(self.clip_sample), **kw)

    def sample_prev_timestep(self, xt, noise_pred, t, z=None, step_index=None):
        """(x_prev, x0) from (x_t, eps, t) for a timestep t of the schedule, shaped like
        LinearNoiseScheduler.sample_prev_timestep.  The noise is `z` when given, otherwise the fused Philox stream
        keyed by (self.seed, step, element); step defaults to t's position in timesteps(), the step index
        sampler.DDPMSampler uses, so a loop over timesteps() draws the sampler's noise."""
        xt, noise_pred, z = step_inputs(xt, noise_pred, z)
        ts, k = self._position(t)
        coef = self.coef_table(xt.device)[ts[k]]
        return self.update(xt, noise_pred, coef, z=z, want_x0=True, seed=self.seed,
                           step=k if step_index is None else int(step_index))
