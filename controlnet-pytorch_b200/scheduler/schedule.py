"""The strided timestep schedules the few-step samplers (ddim_scheduler.py, dpm_solver_scheduler.py) share, and the
truncated ("tail") schedules of image-to-image sampling that every scheduler shares."""
import math
import numbers
from fractions import Fraction

import torch

from .. import runtime as rt

SPACINGS = ("trailing", "leading")


def strided_timesteps(owner, T, num_inference_steps, spacing, explicit=None, steps=None):
    """tau_0 > ... > tau_{S-1} as a tuple of ints.  The schedule is `explicit` when given (strictly decreasing, inside
    [0, T)), otherwise S = `steps` (or `num_inference_steps`) timesteps with the given spacing:
      "trailing": round(T - k T / S) - 1, k = 0 .. S-1 (round half to even), starting at T-1 where x_T ~ N(0, I);
      "leading":  (S-1-k) * (T // S), ending at 0.
    `owner` names the scheduler in the error messages."""
    if explicit is not None:
        ts = explicit
        if steps is not None and int(steps) != len(ts):
            raise rt.CnbError(f"{owner}: steps={steps} disagrees with the {len(ts)} explicit timesteps")
        if not ts or any(not 0 <= t < T for t in ts) or any(a <= b for a, b in zip(ts, ts[1:])):
            raise rt.CnbError(f"{owner}: timesteps must be strictly decreasing and inside [0, {T})")
        return ts
    S = num_inference_steps if steps is None else steps
    if isinstance(S, bool) or not isinstance(S, numbers.Integral) or not 1 <= S <= T:
        raise rt.CnbError(f"{owner}: the number of steps must be an int in [1, {T}] (got {S!r})")
    if spacing == "trailing":
        return tuple(round(Fraction(T) - Fraction(k * T, S)) - 1 for k in range(S))   # round(): half to even
    if spacing == "leading":
        return tuple((S - 1 - k) * (T // S) for k in range(S))
    raise rt.CnbError(f"{owner}: spacing must be one of {SPACINGS} (got {spacing!r})")


def tail(owner, ts, skip):
    """The schedule `ts` without its first `skip` timesteps, 0 <= skip < len(ts); skip = 0 returns `ts` itself."""
    if isinstance(skip, numbers.Integral) and not isinstance(skip, bool) and skip == 0:
        return ts
    if isinstance(skip, bool) or not isinstance(skip, numbers.Integral) or not 0 <= skip < len(ts):
        raise rt.CnbError(f"{owner}: skip must be an int in [0, {len(ts)}) for a schedule of {len(ts)} steps "
                          f"(got {skip!r})")
    return ts[int(skip):]


def strength_to_skip(S, strength):
    """The number of leading timesteps image-to-image sampling skips in a schedule of S steps at `strength` in (0, 1]:
    it keeps n = min(S, int(S * strength)) steps, the rule of diffusers' img2img pipelines, and returns S - n.
    int() truncates the float product, so a strength that is not a multiple of 1 / S in binary keeps one step fewer
    than the decimal suggests: int(100 * 0.29) is int(28.999999999999996) = 28, while int(50 * 0.6) = 30."""
    if isinstance(strength, bool) or not isinstance(strength, numbers.Real) or not math.isfinite(strength) or \
            not 0.0 < strength <= 1.0:
        raise rt.CnbError(f"strength must be a finite number in (0, 1] (got {strength!r})")
    n = min(S, int(S * float(strength)))
    if n == 0:
        raise rt.CnbError(f"strength={strength!r} keeps no step of a schedule of S={S} steps (int(S * strength) = 0)")
    return S - n


def noise_levels(base, ts):
    """fp32 [len(ts), 2]: row k is (sqrt_alpha_cum_prod[tau_{k+1}], sqrt_one_minus_alpha_cum_prod[tau_{k+1}]) of the
    LinearNoiseScheduler `base`, the last row (1, 0).  After step k the known region of an inpainting run is
    base.add_noise(x_ref, z, tau_{k+1}) bit for bit, and after the last step it is x_ref exactly."""
    nxt = list(ts[1:])
    lv = torch.empty((len(ts), 2), dtype=torch.float32)
    lv[:-1, 0] = base.sqrt_alpha_cum_prod[nxt]
    lv[:-1, 1] = base.sqrt_one_minus_alpha_cum_prod[nxt]
    lv[-1, 0], lv[-1, 1] = 1.0, 0.0
    return lv
