"""The strided timestep schedules the few-step samplers (ddim_scheduler.py, dpm_solver_scheduler.py) share."""
import numbers
from fractions import Fraction

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
