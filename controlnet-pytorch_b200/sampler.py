"""Sampling drivers for the hot path: the timestep loop of tools/sample_ddpm_controlnet.py:43-51 /
tools/sample_ldm_controlnet.py:45-50 with the per-step host work removed.

  * one denoising step (sampler prologue -> ControlNet forward -> fused scheduler update -> step counter bump) is
    captured ONCE into a CUDA graph and replayed for every timestep: t, the scheduler coefficients and the Philox
    step are read from device memory, so there is no H2D copy, no host sync and no CPU RNG inside the loop;
  * noise is Philox keyed by the GLOBAL element index, so the result is independent of how the batch is sharded;
  * data parallel: each rank owns a contiguous slice of the batch, no collective inside the loop, one all_gather of
    the final samples (NCCL over NVLink) at the end.

The algorithm is the scheduler's: a LinearNoiseScheduler (DDPM, t = steps-1 .. 0), a DDIMScheduler or a
DPMSolverMultistepScheduler (strided schedules) answers the same questions - `timesteps(steps)`, the [T, 6]
`coef_table(device, steps)` the sampler prologue reads at row t, the fused `update` launch, the `graph_key(steps)` of
what a captured step depends on, and `new_state(x)`, the dict of per-run device buffers carried from one step to the
next (DPM-Solver++'s previous data prediction; empty for DDPM and DDIM) that the sampler allocates once per run, or
once per captured graph, and passes to every `update`.  With steps=None the schedule is the scheduler's own (all T
timesteps for DDPM, num_inference_steps for the strided schedulers).

Image-to-image and inpainting (`img2img`) run the tail of the schedule, `timesteps(steps, skip)` with
skip = strength_to_skip(S, strength), from the reference noised to its first timestep (cnb_add_noise, outside the
graph).  With a mask the captured step gains one launch after the update, cnb_inpaint_blend, which puts the known
region back at the noise level of the next timestep.  The noise z of the start and of every blend is the x_T stream
(seed, _XT_STEP, global element): fixed over the run, like diffusers' legacy inpainting, and drawn in the kernels.

Control strength (`control=ControlOptions(...)`, a ControlNet only): a conditioning scale on the zero convolutions, a
window [start, end) of the schedule outside which the step is the frozen U-Net alone, and hint guidance
eps = eu + w * (ec - eu).  A non-default `control` captures up to two step graphs over the same sampler-owned buffers,
the control graph (prologue -> model._forward_controlled -> update -> [blend] -> bump) and the plain graph (prologue ->
model.trained_unet -> update -> [blend] -> bump), and picks one per step on the host from `ControlOptions.keep`.

Each call is checked and set up once, by `DDPMSampler._plan`, whichever loop runs it.  Both loops run one step body,
`DDPMSampler._step` (forward -> update -> [blend]): the eager loop with host values, the captured step between the
prologue and the bump with the device step counter and the sampler-owned buffers.
"""

import collections
import dataclasses
import math
import numbers

import torch

from . import ops
from . import runtime as rt
from .models import _engine as E
from .scheduler.schedule import noise_levels, strength_to_skip

_XT_STEP = (1 << 40)   # Philox "step" reserved for drawing x_T


@dataclasses.dataclass(frozen=True)
class ControlOptions:
    """How strongly the hint steers a ControlNet sample (diffusers' names in brackets):
      scale     multiplies every down and mid zero-convolution residual (controlnet_conditioning_scale); the hint
                block's own zero convolution is not scaled;
      start/end the control branch runs on the steps i of the n steps run with not (i / n < start or
                (i + 1) / n > end) (control_guidance_start / _end); the other steps are the frozen U-Net alone;
      guidance  w of eps = eu + w * (ec - eu), ec the ControlNet's and eu the frozen U-Net's prediction (guidance_scale
                with guess_mode and no prompt); 1 is no guidance.
    ControlOptions() is the plain ControlNet sampler."""
    scale: float = 1.0
    start: float = 0.0
    end: float = 1.0
    guidance: float = 1.0

    def __post_init__(self):
        for name in ("scale", "start", "end", "guidance"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(v):
                raise rt.CnbError(f"ControlOptions: {name} must be a finite number (got {v!r})")
        for name in ("scale", "guidance"):
            if getattr(self, name) < 0:
                raise rt.CnbError(f"ControlOptions: {name} must be >= 0 (got {getattr(self, name)!r})")
        if not 0 <= self.start < self.end <= 1:
            raise rt.CnbError(f"ControlOptions: need 0 <= start < end <= 1 (got start={self.start!r}, "
                              f"end={self.end!r})")

    def keep(self, n):
        """Per step of the n steps run (the tail for img2img): True where the control branch runs.  All False when
        scale or guidance is 0: eps is then exactly the frozen U-Net's."""
        if self.scale == 0 or self.guidance == 0:
            return [False] * n
        return [not (i / n < self.start or (i + 1) / n > self.end) for i in range(n)]


# One sampling call, checked and derived once by DDPMSampler._plan: the timesteps run (img2img's tail), the scheduler's
# [T, 6] coefficient table on x's device, the checked ControlOptions and its window keep(len(ts)) (both None for the
# plain ControlNet step), img2img's checked reference and mask and the blend's noise-level table (None without a mask),
# and the key of everything a captured step depends on: an equal key reuses the captured graph(s).
_Plan = collections.namedtuple("_Plan", "ts table ctl keep x_ref mask levels key")


class DDPMSampler:
    def __init__(self, model, scheduler, seed=0, use_graph=True):
        self.model, self.scheduler, self.seed, self.use_graph = model, scheduler, int(seed), use_graph
        self._graph = None
        self._key = None

    # ---- x_T -------------------------------------------------------------------------------------------
    def draw_xT(self, shape, device, elem_offset=0):
        return ops.philox_normal(shape, device, self.seed, _XT_STEP, elem_offset)

    # ---- what both loops share: the checked run of one call, the image-to-image start, the step body --------
    def _base(self):
        """The LinearNoiseScheduler whose tables define the noise levels (a strided scheduler's `base`)."""
        return getattr(self.scheduler, "base", self.scheduler)

    def _noised_start(self, x_ref, t, z, elem_offset, out=None):
        """add_noise(x_ref, z, t) with the base scheduler's fp32 values at t; z=None is the x_T stream."""
        b = self._base()
        return ops.add_noise(x_ref, float(b.sqrt_alpha_cum_prod[t]), float(b.sqrt_one_minus_alpha_cum_prod[t]), z=z,
                             seed=self.seed, step=_XT_STEP, elem_offset=elem_offset, out=out)

    def _plan(self, x_T, hint, steps, elem_offset, x_ref=None, mask=None, strength=1.0, control=None):
        """Every check of a sampling call and what it runs (_Plan).  With x_ref the run is img2img and x_T, when given,
        the eager loop's injected noise: x_ref contiguous fp32 NCHW, the mask fp32 (bool converted once),
        [B, 1 or C, H, W] with values in [0, 1] (one check per call, outside the loop), skip from strength.  The hint
        must have the batch size of the x the model reads: the forward's convolutions index the hint by sample."""
        rt.require_cuda(x_T, hint, x_ref, mask)
        sch, skip = self.scheduler, 0
        if x_ref is not None:
            if x_ref.dtype != torch.float32 or x_ref.dim() != 4:
                raise rt.CnbError("img2img: the reference must be a fp32 NCHW tensor")
            x_ref = x_ref.contiguous()
            skip = strength_to_skip(len(sch.timesteps(steps)), strength)
        if mask is not None:
            if x_ref is None:
                raise rt.CnbError("a mask needs the reference x_ref")
            if mask.dtype == torch.bool:
                mask = mask.float()
            B, C, H, W = x_ref.shape
            if mask.dtype != torch.float32 or mask.dim() != 4 or tuple(mask.shape) not in ((B, 1, H, W), (B, C, H, W)):
                raise rt.CnbError(f"img2img: the mask must be fp32 or bool, shaped [{B}, 1 or {C}, {H}, {W}] "
                                  f"(got {mask.dtype} {tuple(mask.shape)})")
            mask = mask.contiguous()
            if not bool(((mask >= 0) & (mask <= 1)).all()):
                raise rt.CnbError("img2img: mask values must lie in [0, 1] (1 = generate, 0 = keep the reference)")
        x = x_T if x_ref is None else x_ref
        if hint.shape[0] != x.shape[0]:
            raise rt.CnbError(f"the hint's batch size {hint.shape[0]} differs from the {x.shape[0]} samples of "
                              f"{'x_T' if x_ref is None else 'x_ref'}")
        if control is not None and not isinstance(control, ControlOptions):
            raise rt.CnbError(f"control must be a sampler.ControlOptions (got {type(control).__name__})")
        ctl = None if control is None or control == ControlOptions() else control     # None: the plain step
        if ctl is not None and not hasattr(self.model, "_forward_controlled"):
            raise rt.CnbError(f"control options need a ControlNet; {type(self.model).__name__} has no control branch")
        ts = sch.timesteps(steps, skip)
        table = sch.coef_table(x.device, steps, skip)
        keep = None if ctl is None else ctl.keep(len(ts))
        levels = None if mask is None else noise_levels(self._base(), ts).to(x.device)
        # the table's address tells apart schedulers with equal graph keys but other beta schedules; the noise-level
        # table is sampler-owned and refreshed on reuse, so its values need no key
        key = (tuple(x.shape), tuple(hint.shape), sch.graph_key(steps, skip), table.data_ptr(), elem_offset,
               rt.get_mode(), str(x.device), self._param_stamp(), skip, None if mask is None else tuple(mask.shape))
        if ctl is not None:
            key += ((ctl.scale, ctl.guidance, tuple(keep)),)
        return _Plan(ts, table, ctl, keep, x_ref, mask, levels, key)

    def _step(self, ctl, controlled, hint, xt, t, coef, state, blend, elem_offset, step=0, step_dev=None, z=None,
              z0=None, out=None, x0_out=None):
        """One denoising step, the body of both loops; returns (x, x0).  eps is the model's forward (ctl None), its
        controlled forward or, outside the control window, the frozen U-Net alone; then the scheduler's fused update
        and, with blend = (x_ref, mask, levels), the inpainting blend.  The eager loop passes host values (step=k,
        injected z and z0), the captured step the device step counter and the sampler-owned buffers."""
        if ctl is None:
            eps = self.model(xt, t, hint)
        elif controlled:
            eps = self.model._forward_controlled(xt, t, hint, ctl.scale,
                                                 None if ctl.guidance == 1.0 else float(ctl.guidance))
        else:
            eps = self.model.trained_unet(xt, t)
        xt, x0 = self.scheduler.update(xt, eps, coef, z=z, seed=self.seed, step=step, step_dev=step_dev,
                                       elem_offset=elem_offset, out=out, x0_out=x0_out, **state)
        if blend is not None:
            ops.inpaint_blend(xt, *blend, step=step, step_dev=step_dev, z=z0, seed=self.seed, noise_step=_XT_STEP,
                              elem_offset=elem_offset)
        return xt, x0

    # ---- eager loop (injected z, parity tests, per-step callbacks) ----------------------------------------
    @torch.no_grad()
    def sample_eager(self, x_T, hint, steps=None, zs=None, elem_offset=0, callback=None, x_ref=None, mask=None,
                     strength=1.0, control=None):
        """The loop without a graph; returns (x, x0).  With `x_ref` it is img2img's loop (see there): it starts from
        add_noise(x_ref, z, tau_skip) and, with `mask`, blends after every step, where z is x_T when given (injected
        noise) and otherwise the x_T stream.  `control`: ControlOptions (see there)."""
        p = self._plan(x_T, hint, steps, elem_offset, x_ref, mask, strength, control)
        z0 = None if x_ref is None or x_T is None else x_T.contiguous()
        xt = x_T.contiguous() if x_ref is None else self._noised_start(p.x_ref, p.ts[0], z0, elem_offset)
        blend = None if p.mask is None else (p.x_ref, p.mask, p.levels)
        x0 = None
        state = self.scheduler.new_state(xt)
        t_dev = torch.empty((1,), device=xt.device, dtype=torch.int64)
        for k, t in enumerate(p.ts):
            t_dev.fill_(t)
            # the last step adds no noise in any scheduler, so zs may stop one short of the schedule
            z = zs[k].to(xt.device) if (zs is not None and k < len(p.ts) - 1) else None
            xt, x0 = self._step(p.ctl, p.keep is None or p.keep[k], hint, xt, t_dev, p.table[t], state, blend,
                                elem_offset, step=k, z=z, z0=z0)
            if callback is not None:
                callback(t, xt, x0)
        return xt, x0

    # ---- graph-replayed loop ----------------------------------------------------------------------------
    def _param_stamp(self):
        """(version, address) of every parameter: a load_state_dict / optimizer step / .to() after capture changes it,
        and the graph (which baked the packed-weight caches derived from the old values) is rebuilt."""
        return tuple((p._version, p.data_ptr()) for p in self.model.parameters())

    def _refresh_hint(self):
        """The captured step reads the hint FEATURE tensors the warm-up cached (models/_engine.HintCache); after the
        static hint buffer has been overwritten they are recomputed in place, outside the graph, once per call."""
        fn = getattr(self.model, "_hint_feat", None)
        if fn is None:
            return
        fn(self._hint, rt.get_mode())

    def _capture(self, x_T, hint, steps, elem_offset, plan=None):
        """Capture the step graph(s) of `plan` (by default the plain run of x_T, hint and steps) over buffers the
        sampler owns, x_T's copy the start of the run."""
        p = self._plan(x_T, hint, steps, elem_offset) if plan is None else plan
        dev = x_T.device
        self.xt = x_T.clone().contiguous()
        # the graph reads a hint buffer OWNED by the sampler: callers may free or overwrite theirs
        self._hint = hint.clone().contiguous()
        hint = self._hint
        self.x0 = torch.empty_like(self.xt)
        self.t_seq = torch.tensor(p.ts, dtype=torch.int64).to(dev)
        self.step_idx = torch.zeros((1,), device=dev, dtype=torch.int32)
        self.t_out = torch.zeros((1,), device=dev, dtype=torch.int64)
        self.coef = torch.zeros((6,), device=dev, dtype=torch.float32)
        self._table = p.table        # the graph reads it: kept alive, so no other table can take its address
        self._state = self.scheduler.new_state(self.xt)   # carried across replays: owned by the sampler, as the graph
        # inpainting: the reference and the mask the blend reads, owned like the hint, and the plan's own level table
        self._blend = None if p.mask is None else (p.x_ref.clone(), p.mask.clone(), p.levels)
        L = rt.lib()

        def one_step(controlled):
            rt.check(L.cnb_sampler_prologue(self.step_idx.data_ptr(), self.t_seq.data_ptr(), self.t_out.data_ptr(),
                                            p.table.data_ptr(), self.coef.data_ptr(), rt.stream()))
            self._step(p.ctl, controlled, hint, self.xt, self.t_out, self.coef, self._state, self._blend, elem_offset,
                       step_dev=self.step_idx, out=self.xt, x0_out=self.x0)
            rt.check(L.cnb_bump_index(self.step_idx.data_ptr(), 1, rt.stream()))

        def capture(controlled):
            # warm-up on a side stream: builds weight / hint caches and sets kernel attributes outside the capture
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self.step_idx.zero_()
                one_step(controlled)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize(dev)
            c0 = rt.launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                one_step(controlled)
            return g, rt.launch_count() - c0

        # with control options, the control graph and the plain graph share every buffer above and are captured only
        # when some step uses them; replay_steps picks one per step from self._keep
        self._keep = p.keep
        self._graphs = {}
        self.launches_per_step = self.plain_launches_per_step = None
        for controlled in ((True,) if p.keep is None else sorted(set(p.keep), reverse=True)):
            g, n = capture(controlled)
            self._graphs[controlled] = g
            if controlled:
                self.launches_per_step = n
            else:
                self.plain_launches_per_step = n
        self._graph = self._graphs[True] if self._keep is None else self._graphs[self._keep[0]]
        self._nsteps, self._pos = len(p.ts), 0
        # keep every tensor the graphs read alive for as long as the graphs: the hint features (HintCache may evict)
        # and the scaled zero-convolution weights (replaced when another scale is used)
        cache = getattr(self.model, "_hint_cache", None)
        self._baked = (cache.pinned() if cache is not None else []) + E.pinned_scaled(self.model)

    @torch.no_grad()
    def sample(self, x_T, hint, steps=None, elem_offset=0, control=None):
        """Run the scheduler's timesteps (DDPM: t = steps-1 .. 0, SURVEY.md 3.5 semantics) with fused on-device noise;
        returns (x after the last step, x0).  `control`: ControlOptions (see there)."""
        if not self.use_graph:
            return self.sample_eager(x_T, hint, steps, None, elem_offset, control=control)
        plan = self._plan(x_T, hint, steps, elem_offset, control=control)
        self._prepare(x_T, hint, elem_offset, plan)
        self.xt.copy_(x_T)
        return self._run()

    def _prepare(self, x_T, hint, elem_offset, plan):
        """Capture the step graph(s) of `plan`, or refresh the sampler-owned buffers of the ones whose key it has."""
        if self._graph is None or plan.key != self._key:
            self._capture(x_T, hint, None, elem_offset, plan)
            self._key = plan.key
        else:
            self._hint.copy_(hint)
            self._refresh_hint()
            if plan.mask is not None:
                for buf, new in zip(self._blend, (plan.x_ref, plan.mask, plan.levels)):
                    buf.copy_(new)

    def _run(self):
        self.replay_steps(self._nsteps, reset=True)
        out = self.xt.clone(), self.x0.clone()
        check_device_errors()
        return out

    @torch.no_grad()
    def img2img(self, x_ref, hint, strength=1.0, mask=None, steps=None, elem_offset=0, control=None):
        """Image-to-image (SDEdit) and inpainting under the hint; returns (x, x0).
        The run keeps the last n = min(S, int(S * strength)) of the S timesteps of `timesteps(steps)`
        (scheduler.schedule.strength_to_skip) and starts from add_noise(x_ref, z, tau_skip), z the x_T stream
        (seed, _XT_STEP, global element index); step k of the tail draws its noise like step k of a plain run over the
        same tail.  `mask` ([B, 1 or C, H, W], fp32 or bool; 1 = generate, 0 = keep the reference) adds one launch to
        the captured step: after step k the elements with m = 0 are add_noise(x_ref, z, tau_{k+1}) with the same z,
        x_ref exactly after the last step, and soft values blend m * x + (1 - m) * known.  The returned x is blended;
        x0 is the update's own prediction of the last step, before the blend.  `control`: ControlOptions, whose window
        applies to the steps run."""
        if not self.use_graph:
            return self.sample_eager(None, hint, steps, None, elem_offset, x_ref=x_ref, mask=mask, strength=strength,
                                     control=control)
        plan = self._plan(None, hint, steps, elem_offset, x_ref, mask, strength, control)
        self._prepare(plan.x_ref, hint, elem_offset, plan)
        self._noised_start(plan.x_ref, plan.ts[0], None, elem_offset, out=self.xt)
        return self._run()

    def replay_steps(self, n, reset=True):
        """bench.py hook: replay the captured step n times (state continues from wherever it is)."""
        if reset:
            self.step_idx.zero_()
            self._pos = 0
        for _ in range(n):
            if self._pos >= self._nsteps:      # wrap around the schedule instead of running off the t table
                self.step_idx.zero_()
                self._pos = 0
            (self._graph if self._keep is None else self._graphs[self._keep[self._pos]]).replay()
            self._pos += 1


class LDMSampler(DDPMSampler):
    """tools/sample_ldm_controlnet.py:21-64: the same timestep loop on VAE latents, then `vae.decode` of the final
    latents only (:51-53), clamp to [-1, 1] and map to [0, 1] (:57-58).  Decoding runs in chunks so that the
    128x128x256-channel decoder activations of a large batch stay bounded (2.1 GB per 256 samples and tensor)."""

    def __init__(self, model, scheduler, vae, seed=0, use_graph=True, decode_chunk=256):
        super().__init__(model, scheduler, seed=seed, use_graph=use_graph)
        self.vae, self.decode_chunk = vae, int(decode_chunk)

    @torch.no_grad()
    def decode(self, latents, to_unit_range=True):
        rt.require_cuda(latents)
        outs = []
        for lo in range(0, latents.shape[0], self.decode_chunk):
            ims = self.vae.decode(latents[lo:lo + self.decode_chunk].contiguous())
            if to_unit_range:
                ims = (torch.clamp(ims, -1., 1.) + 1) / 2
            outs.append(ims)
        check_device_errors()
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)

    @torch.no_grad()
    def sample_images(self, x_T, hint, steps=None, elem_offset=0, zs=None, to_unit_range=True, control=None):
        """Returns (images, final latents).  zs: injected per-step noise (eager loop, parity tests)."""
        if zs is not None:
            xt, _ = self.sample_eager(x_T, hint, steps, zs, elem_offset, control=control)
        else:
            xt, _ = self.sample(x_T, hint, steps=steps, elem_offset=elem_offset, control=control)
        return self.decode(xt, to_unit_range), xt

    @torch.no_grad()
    def encode_mean(self, images):
        """Latents of images in [-1, 1]: the VAE posterior mean, the first z_channels channels of the encoder output.
        Deterministic, unlike the reference's `encode`, which samples the posterior with CPU noise."""
        rt.require_cuda(images)
        return self.vae._encode_out(images.contiguous(), rt.get_mode())[:, :self.vae.z_channels].contiguous()

    def latent_mask(self, mask, latents):
        """An image-space mask [B, 1, H, W] (fp32 or bool) on the latent grid of `latents`: the maximum over each
        f x f window (cnb_mask_max_pool), so a latent cell touching any repainted pixel is repainted."""
        rt.require_cuda(mask)
        if mask.dtype == torch.bool:
            mask = mask.float()
        if mask.dim() != 4 or mask.shape[0] != latents.shape[0] or mask.shape[1] != 1:
            raise rt.CnbError(f"img2img_images: the image-space mask must be [B, 1, H, W] (got {tuple(mask.shape)})")
        f = mask.shape[2] // latents.shape[2]
        if f < 1 or mask.shape[2] != f * latents.shape[2] or mask.shape[3] != f * latents.shape[3]:
            raise rt.CnbError(f"img2img_images: mask {tuple(mask.shape[2:])} is not a multiple of the latent grid "
                              f"{tuple(latents.shape[2:])}")
        return ops.mask_max_pool(mask.contiguous(), f)

    @torch.no_grad()
    def img2img_images(self, images, hint, strength=1.0, mask=None, steps=None, elem_offset=0, to_unit_range=True,
                       control=None):
        """img2img on the latents of `images` ([-1, 1], encoded to the posterior mean) with an image-space `mask`
        pooled to the latent grid; returns (decoded images, final latents).  The known LATENT region is exact; the
        decoded pixels of the kept region are not (there is no paste-back after decode)."""
        lat = self.encode_mean(images)
        lmask = None if mask is None else self.latent_mask(mask, lat)
        xt, _ = self.img2img(lat, hint, strength=strength, mask=lmask, steps=steps, elem_offset=elem_offset,
                             control=control)
        return self.decode(xt, to_unit_range), xt


class GraphedStudent:
    """Single-step students (tools/sample_consistency_controlnet_distilled.py:60-75,
    tools/sample_distribution_matching_controlnet_distilled.py) replayed from ONE captured CUDA graph per input shape:
    at small batch the forward is ~160 launches of a few microseconds each, so eager Python dispatch (3.9 ms) is the
    whole latency.  The hint block is captured inside the graph (it is part of every call in the reference as well);
    the consistency student's whole-batch early return (`all(sigma <= sigma_min)`, :81-82) is evaluated on the host
    before the replay."""

    def __init__(self, model):
        self.model = model
        self._graphs = {}

    @torch.no_grad()
    def __call__(self, x, t_or_sigma, hint):
        rt.require_cuda(x, hint)
        m = self.model
        cond = torch.as_tensor(t_or_sigma).to(x.device)
        is_sigma = torch.is_floating_point(cond)
        if is_sigma and hasattr(m, "sigma_min") and bool((cond <= m.sigma_min).all()):
            return x
        key = (tuple(x.shape), tuple(hint.shape), tuple(cond.shape), cond.dtype, rt.get_mode(), str(x.device))
        ent = self._graphs.get(key)
        if ent is None:
            sx, sh, sc = x.clone().contiguous(), hint.clone().contiguous(), cond.clone().contiguous()

            def run():
                if hasattr(m, "_hint_cache"):
                    m._hint_cache.clear()              # the hint block must be INSIDE the captured work
                if is_sigma:
                    m._skip_boundary_sync = True
                try:
                    return m(sx, sc, sh)
                finally:
                    if is_sigma:
                        m._skip_boundary_sync = False
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                run()                                   # warm-up: weight caches, kernel attributes
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize(x.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = run()
            if hasattr(m, "_hint_cache"):
                m._hint_cache.clear()                  # the cached feature lives in the graph's private pool
            ent = (g, sx, sc, sh, out)
            self._graphs[key] = ent
        g, sx, sc, sh, out = ent
        sx.copy_(x)
        sc.copy_(cond)
        sh.copy_(hint)
        g.replay()
        res = out.clone()
        check_device_errors()
        return res


def check_device_errors():
    """A bounded mbarrier wait that expired makes a tensor-core kernel drain and leave garbage (csrc/tc_common.cuh); the
    latch is read (and cleared) at the end of every public sampling call so that corrupt samples never return rc = 0."""
    if rt.lib().cnb_tc_error_flag() != 0:
        raise rt.CnbError("a tcgen05 pipeline wait timed out on the device (hang guard): results are invalid")


def shard_bounds(total, world, rank):
    """Contiguous slice [lo, hi) of the batch owned by `rank` (remainder spread over the first ranks)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


@torch.no_grad()
def sample_data_parallel(model, scheduler, shape, hint_fn, steps=None, seed=0, group=None, use_graph=True,
                         gather=True, vae=None, sampler=None, x_T_fn=None, x_ref_fn=None, mask_fn=None, strength=1.0,
                         control=None):
    """One job over all ranks of `group` (tools/sample_ddpm_controlnet.py:21-51 sharded over the GPUs of a box): rank r
    draws (or receives) and denoises samples [lo, hi) of the global batch `shape[0]`, no collective inside the
    timestep loop, and the final samples are all-gathered ONCE (NCCL over NVLink).
    `hint_fn(lo, hi)` returns this shard's hint tensor on the local device (it may do the host -> device copy);
    `x_T_fn(lo, hi)`, when given, supplies the shard's initial noise the same way (the reference draws x_T on the host,
    :26-29); otherwise x_T is Philox noise keyed by the GLOBAL element index, independent of the number of ranks.
    `sampler` re-uses a DDPMSampler / LDMSampler (and its captured step graph) across calls.  With `vae` the shard's
    final latents are decoded locally (LDM path) and the images are what is gathered.
    `x_ref_fn(lo, hi)` (and `mask_fn(lo, hi)`), mirroring hint_fn, make the job img2img (inpainting) at `strength`:
    they return the shard's references and masks, images and image-space masks with `vae` (encoded locally).
    `control`: ControlOptions (see there) for every shard."""
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = shape[0]
    lo, hi = shard_bounds(B, world, rank)
    per = 1
    for d in shape[1:]:
        per *= d
    dev = torch.device("cuda", torch.cuda.current_device())
    smp = sampler
    if smp is None:
        smp = (DDPMSampler(model, scheduler, seed=seed, use_graph=use_graph) if vae is None else
               LDMSampler(model, scheduler, vae, seed=seed, use_graph=use_graph))
    if x_T_fn is not None and x_ref_fn is not None:
        raise rt.CnbError("sample_data_parallel: x_T_fn and x_ref_fn exclude each other (img2img starts from x_ref)")
    if mask_fn is not None and x_ref_fn is None:
        raise rt.CnbError("sample_data_parallel: mask_fn needs x_ref_fn")
    kw = dict(steps=steps, elem_offset=lo * per, control=control)
    if x_ref_fn is not None:                   # xt: with vae the shard's decoded images
        mask = None if mask_fn is None else mask_fn(lo, hi)
        run = smp.img2img if vae is None else smp.img2img_images
        xt, _ = run(x_ref_fn(lo, hi), hint_fn(lo, hi), strength=strength, mask=mask, **kw)
    else:
        x_T = x_T_fn(lo, hi) if x_T_fn is not None else smp.draw_xT((hi - lo,) + tuple(shape[1:]), dev, lo * per)
        run = smp.sample if vae is None else smp.sample_images
        xt, _ = run(x_T, hint_fn(lo, hi), **kw)
    if not gather or world == 1:
        return xt
    return gather_shards(xt, B, group)


def gather_shards(x_local, total, group=None):
    """The one exchange step of the job: concatenate every rank's contiguous batch shard (shard_bounds order).
    all_gather_into_tensor when the shards are equal, padded all_gather otherwise.  Backend-agnostic (NCCL on the
    GPUs; the world_size-2 gloo test drives it on CPU tensors)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    sizes = [b - a for a, b in (shard_bounds(total, world, r) for r in range(world))]
    tail = tuple(x_local.shape[1:])
    x_local = x_local.contiguous()
    if all(n == sizes[0] for n in sizes):
        out = torch.empty((total,) + tail, device=x_local.device, dtype=x_local.dtype)
        dist.all_gather_into_tensor(out, x_local, group=group)
        return out
    mx = max(sizes)
    padded = torch.zeros((mx,) + tail, device=x_local.device, dtype=x_local.dtype)
    padded[: x_local.shape[0]] = x_local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:n] for p, n in zip(parts, sizes)], dim=0)
