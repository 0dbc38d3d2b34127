"""DPM-Solver++ multistep sampling (scheduler/dpm_solver_scheduler.py, cnb_dpm_solver_step).

CPU: the schedules and the rejection of bad arguments, the [T, 6] coefficient table against an independent float64
restatement, the order-1 rows against DDIM's (eta = 0 for "ode", eta = 1 for "sde"), and the convergence orders of
DDIM and 2M on an analytic Gaussian model whose exact ODE solution is known.  GPU: the fused kernel against a torch-CPU
fp32 restatement of its operation order (bit for bit), the history buffer untouched by first-order rows, the order-1
samplers against DDIM, the convergence orders through the graph-replayed sampler, graph replay against the eager loop,
sharding, re-capture and the hand-written loop of sample_prev_timestep.  Parity of the trajectory with the oracle for
the DDPM and the LDM ControlNet and the MNIST-size launch count run in test_ddim.py, for DDIM and DPM-Solver++ alike.
"""
import pytest
import torch

from helpers import (rel_l2, syn, _base, _ddim, _dpm, _dpm_rows, _fill, _hang_guard, _mod,
                     rt)  # noqa: F401 (fixtures)

MU, SD = 0.3, 0.5                           # the analytic model: data ~ N(MU, SD^2), element-wise
CONV_TS = {S: tuple(999 - k * (900 // S) for k in range(S + 1)) for S in (9, 18, 36)}   # S steps from 999 to 99


# ---- the analytic model: eps(x, t) and the exact probability-flow ODE solution for Gaussian data --------------------
def _tables64(base):
    return base.sqrt_alpha_cum_prod.double(), base.sqrt_one_minus_alpha_cum_prod.double()


def _eps(x, a, s):
    return s * (x - a * MU) / (a * a * SD * SD + s * s)


def _exact(base, x_T, ts):
    """The data prediction at ts[-1] of the exact ODE solution through x_T at ts[0]."""
    sa, s1m = _tables64(base)
    a0, s0, a1, s1 = sa[ts[0]], s1m[ts[0]], sa[ts[-1]], s1m[ts[-1]]
    c = (x_T - a0 * MU) / torch.sqrt(a0 ** 2 * SD ** 2 + s0 ** 2)
    x = a1 * MU + c * torch.sqrt(a1 ** 2 * SD ** 2 + s1 ** 2)
    return (x - s1 * _eps(x, a1, s1)) / a1


def _host_solve(base, table, ts, x_T, kind):
    """The table's linear form in float64 on the analytic model: "dpm" rows (x, D, D_prev) or "ddim" rows (x0, eps)."""
    sa, s1m = _tables64(base)
    x, d_prev = x_T.double(), None
    for t in ts:
        c = table[t].double()
        e = _eps(x, sa[t], s1m[t])
        d = (x - c[0] * e) / c[1]
        if kind == "ddim":
            x = c[2] * d + c[3] * e
        else:
            x = c[2] * x + c[3] * d + (c[4] * d_prev if c[4] != 0 else 0.0)
        d_prev = d
    return x


def _errors(kind, x_T):
    base, out = _base(), {}
    for S, ts in CONV_TS.items():
        s = _ddim(base, timesteps=ts) if kind == "ddim" else _dpm(base, timesteps=ts)
        got = _host_solve(base, s.coef_table_host(), ts, x_T, kind)
        out[S] = rel_l2(got, _exact(base, x_T.double(), ts))
    return out


def _check_orders(ddim, dpm):
    for S in (9, 18):
        assert 1.8 <= ddim[S] / ddim[2 * S] <= 2.2, (S, ddim)
        assert dpm[S] / dpm[2 * S] >= 3.5, (S, dpm)
    assert dpm[18] < 0.25 * ddim[18], (ddim, dpm)


# ---- CPU ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 20, 50, 1000])
def test_timesteps_are_the_ddim_schedules(S):
    for spacing in ("trailing", "leading"):
        want = _ddim(num_inference_steps=S, spacing=spacing).timesteps()
        assert _dpm(num_inference_steps=S, spacing=spacing).timesteps() == want
        assert _dpm(num_inference_steps=7, spacing=spacing).timesteps(S) == want
    assert _dpm(timesteps=[9, 4, 0]).timesteps(3) == (9, 4, 0)


def test_bad_arguments_are_rejected():
    CnbError = _mod("runtime").CnbError
    for kw in (dict(order=0), dict(order=3), dict(order=True), dict(order=1.5), dict(variant="sdeint"),
               dict(variant=None), dict(num_inference_steps=0), dict(num_inference_steps=1001),
               dict(num_inference_steps=2.5), dict(spacing="linspace"), dict(timesteps=[3, 3, 1]),
               dict(timesteps=[1, 2]), dict(timesteps=[1000, 5]), dict(timesteps=[5, -1]), dict(timesteps=[])):
        with pytest.raises(CnbError):
            _dpm(**kw)
    with pytest.raises(CnbError):
        _dpm(timesteps=[9, 4, 0]).timesteps(4)
    for attr, bad in (("order", 3), ("variant", "euler"), ("spacing", "x"), ("num_inference_steps", 0)):
        s = _dpm()
        setattr(s, attr, bad)                                          # attributes are re-validated on use
        with pytest.raises(CnbError):
            s.coef_table_host()
        with pytest.raises(CnbError):
            s.graph_key()


@pytest.mark.parametrize("ldm", [False, True])
@pytest.mark.parametrize("S,order,variant,spacing", [(20, 2, "ode", "trailing"), (20, 2, "sde", "trailing"),
                                                     (7, 1, "ode", "leading"), (10, 1, "sde", "leading"),
                                                     (2, 2, "ode", "trailing"), (1, 2, "sde", "trailing")])
def test_coef_table_matches_the_restated_contract(ldm, S, order, variant, spacing):
    base = _base(ldm)
    s = _dpm(base, num_inference_steps=S, order=order, variant=variant, spacing=spacing)
    ts = s.timesteps()
    tab = s.coef_table_host()
    assert tab.shape == (1000, 6) and tab.dtype == torch.float32
    ddpm = base.coef_table_host()
    on = torch.zeros(1000, dtype=torch.bool)
    on[list(ts)] = True
    assert torch.isnan(tab[~on]).all()                                # off-schedule rows poison the output
    for t, row in _dpm_rows(base, ts, order, variant).items():
        assert torch.equal(tab[t], torch.tensor(row, dtype=torch.float64).float()), t
        assert torch.equal(tab[t, :2], ddpm[t, :2]), t                # the DDPM table's fp32 values, bit for bit
    assert tab[ts[0], 4] == 0.0 and tab[ts[-1], 4] == 0.0             # no D_{-1}; the last step is first order
    assert tab[ts[-1], 2:].tolist() == [0.0, 1.0, 0.0, 0.0]           # the last step is x = D, without noise
    if order == 1:
        assert (tab[on, 4] == 0).all()
    elif S > 2:
        assert (tab[list(ts[1:-1]), 4] != 0).all()
    assert (tab[on, 5] == 0).all() if variant == "ode" else (tab[list(ts[:-1]), 5] > 0).all()


@pytest.mark.parametrize("ldm", [False, True])
@pytest.mark.parametrize("variant,eta", [("ode", 0.0), ("sde", 1.0)])
def test_order1_rows_are_ddim_rows(ldm, variant, eta):
    """DDIM's x_prev = c2 x0 + c3 eps + c4 z with eps = (x - c1 x0) / c0 is (c3 / c0) x + (c2 - c3 c1 / c0) x0 + c4 z:
    equal within 3 fp32 ulp of the magnitudes combined (DDIM's rounded c0 .. c3 bound the agreement)."""
    base = _base(ldm)
    ulp = 2.0 ** -23
    for S in (20, 50, 1000):
        d = _ddim(base, num_inference_steps=S, eta=eta).coef_table_host().double()
        p = _dpm(base, num_inference_steps=S, order=1, variant=variant).coef_table_host().double()
        for t in _ddim(base, num_inference_steps=S).timesteps():
            x_coef, mix = float(d[t, 3] / d[t, 0]), float(d[t, 3] * d[t, 1] / d[t, 0])
            d_coef = float(d[t, 2]) - mix
            assert abs(float(p[t, 2]) - x_coef) <= 3 * ulp * abs(x_coef), (S, t)
            assert abs(float(p[t, 3]) - d_coef) <= 3 * ulp * (abs(float(d[t, 2])) + abs(mix)), (S, t)
            assert abs(float(p[t, 5] - d[t, 4])) <= 3 * ulp * abs(float(d[t, 4])), (S, t)
            assert p[t, 4] == 0.0


def test_convergence_orders_on_the_analytic_model():
    x_T = torch.randn(20000, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    ddim, dpm = _errors("ddim", x_T), _errors("dpm", x_T)
    _check_orders(ddim, dpm)
    assert 0.05 < ddim[9] < 0.12 and dpm[9] < 0.03 and dpm[36] < 4e-4     # the magnitudes the docs quote


# ---- GPU ---------------------------------------------------------------------------------------------------
def _host_dpm(xt, eps, z, hist, row, clip):
    """The kernel's operation order in torch-CPU fp32, one rounding per operation: (x_prev, x0, D)."""
    c = row.float()
    v = (xt - c[0] * eps) / c[1]
    x0 = torch.clamp(v, -1.0, 1.0)
    d = x0 if clip else v
    p = c[2] * xt + c[3] * d
    if float(c[4]) != 0.0:
        p = p + c[4] * hist
    if float(c[5]) != 0.0:
        p = p + c[5] * z
    return p, x0, d


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["ode", "sde"])
def test_kernel_matches_the_host_restatement_bit_for_bit(rt, variant):
    ops = _mod("ops")
    s = _dpm(num_inference_steps=20, variant=variant)
    ts = s.timesteps()
    tab = s.coef_table_host()
    dtab = s.coef_table("cuda")
    g = torch.Generator().manual_seed(3)
    for n in (4 * 1024, 4 * 257 + 3):
        # scaled up so that clamping to [-1, 1] matters at every row
        xt, eps, z, h = (3 * torch.randn(n, generator=g) for _ in range(4))
        xc, ec, zc = xt.cuda(), eps.cuda(), z.cuda()
        for t in (ts[0], ts[len(ts) // 2], ts[-1]):
            for clip in (False, True):
                want_p, want_x0, want_d = _host_dpm(xt, eps, z, h, tab[t], clip)
                hist = h.cuda()
                p, x0 = ops.dpm_solver_step(xc, ec, dtab[t], z=zc, clip_sample=clip, seed=1, step=2, hist=hist)
                assert torch.equal(p.cpu(), want_p) and torch.equal(x0.cpu(), want_x0), (n, t, clip)
                assert torch.equal(hist.cpu(), want_d), (n, t, clip)
                # out aliasing xt, no x0 output
                buf, hist = xc.clone(), h.cuda()
                q, none = ops.dpm_solver_step(buf, ec, dtab[t], z=zc, want_x0=False, clip_sample=clip, out=buf,
                                              hist=hist)
                assert none is None and q is buf and torch.equal(buf, p) and torch.equal(hist.cpu(), want_d)
        # fused noise at an unaligned global offset, with the tail path, on a second-order row
        t = ts[1]
        assert tab[t, 4] != 0
        for off in (0, 6, 4 * 1001 + 1):
            want = ops.philox_normal((n,), "cuda", 9, 4, elem_offset=off).cpu()
            hist = h.cuda()
            p, _ = ops.dpm_solver_step(xc, ec, dtab[t], z=None, seed=9, step=4, elem_offset=off, hist=hist)
            assert torch.equal(p.cpu(), _host_dpm(xt, eps, want, h, tab[t], False)[0]), (n, off)
            step_dev = torch.tensor([4], dtype=torch.int32, device="cuda")
            hist = h.cuda()
            q, _ = ops.dpm_solver_step(xc, ec, dtab[t], z=None, seed=9, step=0, step_dev=step_dev, elem_offset=off,
                                       hist=hist)
            assert torch.equal(p, q)


@pytest.mark.gpu
def test_first_order_rows_never_read_the_history_and_x0_is_the_ddpm_x0(rt):
    ops = _mod("ops")
    base = _base()
    ddpm = base.coef_table("cuda")
    g = torch.Generator().manual_seed(5)
    n = 4 * 4096 + 1
    xt, eps, z = (torch.randn(n, generator=g).cuda() for _ in range(3))
    for order, variant in ((2, "ode"), (2, "sde"), (1, "ode"), (1, "sde")):
        s = _dpm(base, num_inference_steps=50, order=order, variant=variant)
        ts, tab = s.timesteps(), s.coef_table("cuda")
        for t in (ts if order == 1 else (ts[0], ts[-1])):
            hist = torch.full((n,), float("nan"), device="cuda")
            p, x0 = ops.dpm_solver_step(xt, eps, tab[t], z=z, hist=hist)
            assert torch.isfinite(p).all() and torch.isfinite(hist).all(), (order, variant, t)
            assert torch.equal(x0, ops.sched_step(xt, eps, ddpm[t], z=z)[1]), (order, variant, t)
    CnbError = _mod("runtime").CnbError
    row = _dpm(base).coef_table("cuda")[999]
    for bad in (xt, xt[:n - 1]):                                       # hist aliasing xt; a hist of the wrong size
        with pytest.raises(CnbError):
            ops.dpm_solver_step(xt, eps, row, hist=bad)
    out = torch.empty_like(xt)
    with pytest.raises(CnbError):
        ops.dpm_solver_step(xt, eps, row, out=out, hist=out)


def _tiny(rt):
    rt.set_mode("fp32")
    return _fill(_mod("models.controlnet").ControlNet(syn.TINY_PARAMS)), syn.det_hint(4, 16).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("variant,eta", [("ode", 0.0), ("sde", 1.0)])
def test_order1_sampler_is_the_ddim_sampler(rt, variant, eta):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    dpm = _dpm(num_inference_steps=8, order=1, variant=variant)
    ddim = _ddim(num_inference_steps=8, eta=eta)
    xT = S.DDPMSampler(m, dpm, seed=7).draw_xT((4, 1, 16, 16), "cuda")
    a, a0 = S.DDPMSampler(m, dpm, seed=7).sample(xT, hint)
    b, b0 = S.DDPMSampler(m, ddim, seed=7).sample(xT, hint)
    assert rel_l2(a.cpu(), b.cpu()) < 1e-5 and rel_l2(a0.cpu(), b0.cpu()) < 1e-5


class AnalyticEps(torch.nn.Module):
    """eps(x, t) of data ~ N(MU, SD^2) under the base tables: parameter-free torch ops, which a step graph captures."""

    def __init__(self, base):
        super().__init__()
        self.register_buffer("sa", base.sqrt_alpha_cum_prod.clone())
        self.register_buffer("s1m", base.sqrt_one_minus_alpha_cum_prod.clone())

    def forward(self, x, t, hint):
        a, s = self.sa[t].reshape(-1, 1, 1, 1), self.s1m[t].reshape(-1, 1, 1, 1)
        return s * (x - a * MU) / (a * a * (SD * SD) + s * s)


@pytest.mark.gpu
def test_convergence_orders_through_the_graph_sampler(rt):
    S = _mod("sampler")
    rt.set_mode("fp32")
    base = _base()
    model = AnalyticEps(base).cuda()
    hint = torch.zeros((64, 3, 16, 16), device="cuda")
    xT = S.DDPMSampler(model, base, seed=2).draw_xT((64, 1, 16, 16), "cuda")
    x64 = xT.cpu().double()
    errs = {}
    for kind in ("ddim", "dpm"):
        errs[kind] = {}
        for n, ts in CONV_TS.items():
            s = _ddim(base, timesteps=ts) if kind == "ddim" else _dpm(base, timesteps=ts)
            got, _ = S.DDPMSampler(model, s, seed=2).sample(xT, hint)
            host = _host_solve(base, s.coef_table_host(), ts, x64, kind)
            assert rel_l2(got.cpu().double(), host) < 1e-5, (kind, n)
            errs[kind][n] = rel_l2(got.cpu().double(), _exact(base, x64, ts))
    _check_orders(errs["ddim"], errs["dpm"])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["ode", "sde"])
def test_graph_equals_eager_and_shards_reproduce_the_batch(rt, variant):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    s = _dpm(num_inference_steps=6, variant=variant)
    B, per = 4, 16 * 16
    g = S.DDPMSampler(m, s, seed=11, use_graph=True)
    e = S.DDPMSampler(m, s, seed=11, use_graph=False)
    xT = g.draw_xT((B, 1, 16, 16), "cuda")
    a, a0 = g.sample(xT, hint)
    b, b0 = e.sample(xT, hint)
    assert torch.equal(a, b) and torch.equal(a0, b0)
    assert torch.isfinite(a).all()
    c, c0 = g.sample(xT, hint)                                         # a second replay starts from a fresh history
    assert torch.equal(a, c) and torch.equal(a0, c0)
    x_lo = e.draw_xT((2, 1, 16, 16), "cuda", elem_offset=0)
    x_hi = e.draw_xT((2, 1, 16, 16), "cuda", elem_offset=2 * per)
    c_lo, _ = e.sample(x_lo, hint[:2].contiguous(), elem_offset=0)
    c_hi, _ = e.sample(x_hi, hint[2:].contiguous(), elem_offset=2 * per)
    assert rel_l2(torch.cat([c_lo, c_hi]).cpu(), b.cpu()) < 1e-5
    d = S.sample_data_parallel(m, s, (B, 1, 16, 16), lambda lo, hi: hint[lo:hi], seed=11)
    assert torch.equal(d, a)
    if variant == "ode":
        assert torch.equal(S.DDPMSampler(m, s, seed=12).sample(xT, hint)[0], a)   # no noise: the seed is unused
    else:
        assert not torch.equal(S.DDPMSampler(m, s, seed=12).sample(xT, hint)[0], a)


@pytest.mark.gpu
def test_one_sampler_recaptures_on_every_change(rt):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    s = _dpm(num_inference_steps=5)
    smp = S.DDPMSampler(m, s, seed=4)
    xT = smp.draw_xT((4, 1, 16, 16), "cuda")

    def check(steps=None):
        fresh = _dpm(num_inference_steps=s.num_inference_steps, order=s.order, variant=s.variant,
                     clip_sample=s.clip_sample)
        got, got0 = smp.sample(xT, hint, steps=steps)
        want, want0 = S.DDPMSampler(m, fresh, seed=4).sample(xT, hint, steps=steps)
        assert torch.equal(got, want) and torch.equal(got0, want0)
        return got

    outs = [check()]
    outs.append(check(steps=8))
    s.order = 1
    outs.append(check())
    s.variant = "sde"
    outs.append(check())
    s.order = 2
    outs.append(check())
    s.clip_sample = True
    outs.append(check())
    m.load_state_dict(syn.det_state_dict(m.state_dict(), seed=6))
    outs.append(check())
    for i in range(len(outs) - 1):
        assert not torch.equal(outs[i], outs[i + 1]), i
    # and over to DDIM and DDPM on the same sampler
    ddim = _ddim(s.base, num_inference_steps=5)
    smp.scheduler = ddim
    assert torch.equal(smp.sample(xT, hint)[0], S.DDPMSampler(m, ddim, seed=4).sample(xT, hint)[0])
    smp.scheduler = s.base
    got, _ = smp.sample(xT, hint, steps=5)
    assert torch.equal(got, S.DDPMSampler(m, s.base, seed=4).sample(xT, hint, steps=5)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["ode", "sde"])
def test_sample_prev_timestep_loop_is_the_eager_loop(rt, variant):
    S = _mod("sampler")
    CnbError = _mod("runtime").CnbError
    m, hint = _tiny(rt)
    s = _dpm(num_inference_steps=6, variant=variant)
    s.seed = 13
    xT = S.DDPMSampler(m, s, seed=13).draw_xT((4, 1, 16, 16), "cuda")
    want, want0 = S.DDPMSampler(m, s, seed=13, use_graph=False).sample_eager(xT, hint)
    ts = s.timesteps()
    with torch.no_grad():
        for _ in range(2):                                             # a second loop restarts the history at step 0
            xt = xT
            for t in ts:
                xt, x0 = s.sample_prev_timestep(xt, m(xt, torch.tensor([t], device="cuda"), hint), t)
            assert torch.equal(xt, want) and torch.equal(x0, want0)
        eps = m(xT, torch.tensor([ts[0]], device="cuda"), hint)
        s.sample_prev_timestep(xT, eps, ts[0])
        with pytest.raises(CnbError):
            s.sample_prev_timestep(xT, eps, ts[2])                     # skips step 1
        s.sample_prev_timestep(xT, eps, ts[0])
        with pytest.raises(CnbError):
            s.sample_prev_timestep(xT[:2].contiguous(), eps[:2].contiguous(), ts[1])   # another shape
        s.sample_prev_timestep(xT, eps, ts[0])
        s.sample_prev_timestep(xT, eps, ts[1])
        with pytest.raises(CnbError):
            s.sample_prev_timestep(xT, eps, ts[1])                     # the same step twice
