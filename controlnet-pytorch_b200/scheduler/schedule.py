"""The strided timestep schedules and the scheduler base the few-step samplers (ddim_scheduler.py,
dpm_solver_scheduler.py) share, and what every scheduler shares: the truncated ("tail") schedules of image-to-image
sampling and the input checks of sample_prev_timestep."""
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


def step_inputs(xt, noise_pred, z):
    """The input checks of sample_prev_timestep: xt and noise_pred fp32 CUDA tensors, z a CUDA tensor when given.
    Returns the three made contiguous."""
    rt.require_cuda(xt, noise_pred, z)
    if xt.dtype != torch.float32 or noise_pred.dtype != torch.float32:
        raise rt.CnbError("sample_prev_timestep expects fp32 tensors")
    return xt.contiguous(), noise_pred.contiguous(), None if z is None else z.contiguous()


class StridedScheduler:
    """What DDIMScheduler and DPMSolverMultistepScheduler share: a strided schedule (strided_timesteps) over the
    tables of `base`, a LinearNoiseScheduler; a fp32 [T, 6] coefficient table per schedule, built by the subclass's
    coef_table_host and cached per device; and the graph key.  A subclass sets TAG (the graph key's first element)
    and TAIL_TABLE, and defines _params(): its validated solver parameters, part of both keys."""
    TAG = None
    TAIL_TABLE = False      # True: a tail's rows differ from the full schedule's (coef_table_host takes `skip`)

    def __init__(self, base, num_inference_steps, spacing, clip_sample, timesteps):
        self.base = base
        self.num_timesteps = base.num_timesteps
        self.num_inference_steps, self.spacing, self.clip_sample = num_inference_steps, spacing, clip_sample
        self.explicit_timesteps = None if timesteps is None else tuple(int(t) for t in timesteps)
        self.seed = 0
        self._coef = {}
        self.timesteps()
        self._params()

    def timesteps(self, steps=None, skip=0):
        """tau_0 > ... > tau_{S-1} as a tuple of ints; `steps` overrides num_inference_steps; the tail without the first
        `skip` timesteps (0 <= skip < S) with skip > 0."""
        owner = type(self).__name__
        return tail(owner, strided_timesteps(owner, self.num_timesteps, self.num_inference_steps, self.spacing,
                                             self.explicit_timesteps, steps), skip)

    def coef_table(self, device, steps=None, skip=0):
        """The device copy of coef_table_host.  Without TAIL_TABLE a row depends only on its own timestep and the next
        one, so the tail of `skip` (validated) reads the full schedule's table at the same rows."""
        self.timesteps(steps, skip)
        args = (steps, skip) if self.TAIL_TABLE else (steps,)
        key = (str(device), self.timesteps(*args)) + self._params()
        if key not in self._coef:
            self._coef[key] = self.coef_table_host(*args).to(device)
        return self._coef[key]

    def graph_key(self, steps=None, skip=0):
        """Everything a captured sampling step depends on besides the model and the coefficient table."""
        return (self.TAG, self.timesteps(steps, skip)) + self._params() + (bool(self.clip_sample),)

    def _position(self, t):
        """(timesteps(), k) for the k-th timestep t of the schedule; CnbError for a t off the schedule."""
        ts, ti = self.timesteps(), int(t)
        if ti not in ts:
            raise rt.CnbError(f"{type(self).__name__}: t={ti} is not one of the schedule's timesteps")
        return ts, ts.index(ti)


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
