"""Every production layer across the batch sizes that change its kernel route: float64 values, guard bytes and
bit-for-bit batch invariance.

The library picks a kernel plan from the batch size: for the TMA tcgen05 convolution the halo mode, the N-split
narrowing of BN, two CTAs per SM, resident weights, the grid (and so how many tiles the last round gets) and the
small-tensor im2col descriptor fix-up; for the split-statistics GroupNorm the number of row ranges per sample.  Sharded
sampling gives each rank any number of samples, so every one of these plans runs in production, and DESIGN.md section 5
promises that none of them changes a single bit of any sample.

Here one eager f16 forward of each production workload at B = 2 and B = 1 harvests every layer shape (the call-site
signature without B).  For each convolution shape, cnb_conv2d_route is asked (nothing is launched) for the route at
every B from 1 to the largest batch the workload runs, and the layer is replayed at the batch sizes where the route
changes (both sides of every change), where a CTA first runs a second tile, where the last round first holds a lone
tile, on both sides of the 128 KiB im2col input size, at B = 1 and at the production batches and their 2-, 4- and
8-way shards.  Per-sample operands are periodic (sample b is pool sample b % 5, and 5 divides no tile size), so each
replay must reproduce the canonical B = 5 output bit for bit in every sample, which is itself checked element by
element against float64.  A tile that read a neighbouring sample, a last round that dropped a tile, or an epilogue
whose rounding depends on the plan shows up as a differing sample.
"""
import math
import time

import pytest
import torch

from test_call_sites_gpu import (TAU, WORKLOADS, Recorder, _fill, _gen, _mod, _randn, compare, conv_label,
                                 conv_reference, fill_sentinel, groupnorm_reference, out_window, window_violations)

P = 5                          # pool size of the periodic inputs: divides none of the tile sizes (128 rows, R rows)
IM2COL_SMALL = 131072          # csrc/conv_tma.cu: inputs under this many bytes get the small-tensor descriptor fix-up
SHARDS = (1, 2, 4, 8)


# ---------------------------------------------------------------------------------------------------------------------
# batch-size selection and the periodic comparator (pure, checked on the CPU at the end)
# ---------------------------------------------------------------------------------------------------------------------
def route_class(route):
    """The route without the quantities that grow with every batch size (grid and tile count)."""
    return tuple((k, v) for k, v in route.items() if k not in ("grid", "ntiles"))


def _im2col(route):
    return route["path"] == 2 and not route["halo"]


def _second_round(route):
    return route["ntiles"] > route["grid"] > 0


def pick_batches(routes, in_bytes=(), extra=()):
    """Batch sizes to replay.  routes[i] is the route at B = i + 1; in_bytes the per-sample byte sizes of the inputs
    an im2col route loads; extra the batch sizes always replayed (those above len(routes) are dropped).

    Picks B = 1, the first and last B of every run of one route class, in each run the first B where a CTA runs a
    second tile and the first B where the last round holds a single tile, and for im2col routes the last B whose input
    is under 128 KiB and the next one."""
    n = len(routes)
    picks = {1} | {b for b in extra if 1 <= b <= n}
    lo = 0
    for hi in range(1, n + 1):
        if hi < n and route_class(routes[hi]) == route_class(routes[lo]):
            continue
        picks |= {lo + 1, hi}
        run = range(lo, hi)
        for cond in (_second_round, lambda r: _second_round(r) and r["ntiles"] % r["grid"] == 1):
            b = next((i + 1 for i in run if cond(routes[i])), None)
            if b is not None:
                picks.add(b)
        lo = hi
    for c in in_bytes:
        last = (IM2COL_SMALL - 1) // c
        picks |= {b for b in (last, last + 1) if 1 <= b <= n and _im2col(routes[b - 1])}
    return sorted(picks)


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32}[t.element_size()])


def periodic_mismatch(got, canon):
    """got (B, ...) and canon (P, ...) of one dtype: (sample b, element index) of the first element of got that is not
    bit-equal to canonical sample b % P, else None."""
    g, c = _bits(got), _bits(canon)
    idx = torch.arange(got.shape[0], device=got.device) % canon.shape[0]
    bad = (g != c[idx]).reshape(got.shape[0], -1).any(1)
    if not bool(bad.any()):
        return None
    b = int(bad.nonzero()[0])
    e = (g[b] != c[b % canon.shape[0]]).nonzero()[0]
    return b, tuple(int(v) for v in e)


# ---------------------------------------------------------------------------------------------------------------------
# harvest: every layer shape of the production workloads, with the largest batch it runs at
# ---------------------------------------------------------------------------------------------------------------------
def _shape(rec):
    """The call-site signature without B: per-sample time-embedding tables have B rows."""
    d = {k: v for k, v in rec.items() if k not in ("B", "route")}
    if d.get("temb") and d["temb"][3]:
        d["temb"] = (None,) + tuple(d["temb"][1:])
    return d


def _shard_sizes(batches, bmax):
    shard_bounds = _mod("sampler").shard_bounds
    sizes = set()
    for b in batches:
        for w in SHARDS:
            sizes |= {hi - lo for lo, hi in (shard_bounds(b, w, r) for r in range(w))}
    return {s for s in sizes if 1 <= s <= bmax}


@pytest.fixture(scope="module")
def layers():
    """(ops, rt, convs, groupnorms): {shape key: [shape, Bmax, production batch sizes]}."""
    ops, rt = _mod("ops"), _mod("runtime")
    assert torch.cuda.is_available()
    rt.lib()
    rec = Recorder(ops, rt)
    prev = rt._MODE
    mp = pytest.MonkeyPatch()
    for k in rec.real:
        mp.setattr(ops, k, getattr(rec, k))
    found = {"conv": {}, "groupnorm": {}}
    try:
        rt.set_mode("f16")
        for tag, f16_batches, _, build, call in WORKLOADS:
            bmax = max(f16_batches)
            prod = _shard_sizes(f16_batches, bmax)
            m = _fill(build())
            for B in (2, 1):
                rec.sigs, rec.tag = {}, f"{tag} B={B}"
                with torch.no_grad():
                    call(m, B)
                torch.cuda.synchronize()
                for s in rec.sigs.values():
                    if s["op"] not in found:
                        continue
                    d = _shape(s)
                    e = found[s["op"]].setdefault(tuple(sorted(d.items())), [d, 0, set()])
                    e[1] = max(e[1], bmax)
                    e[2] |= prod
            del m
            torch.cuda.empty_cache()
    finally:
        mp.undo()
        rt._MODE = prev
    print(f"\nlayer shapes: {len(found['conv'])} convolutions, {len(found['groupnorm'])} GroupNorms")
    return ops, rt, found["conv"], found["groupnorm"]


# ---------------------------------------------------------------------------------------------------------------------
# one convolution shape, its operands allocated once at Bmax + 1 samples
# ---------------------------------------------------------------------------------------------------------------------
def _periodic(pool, n):
    return pool[torch.arange(n, device=pool.device) % pool.shape[0]].contiguous()


class ConvLayer:
    """Operands of one harvested convolution shape at Bmax + 1 samples (one guard sample after the largest batch).
    Every per-sample operand (x, x2, the residual, per-sample time-embedding rows) of sample b is pool sample b % P;
    the values are fp16-representable, so every product is exact."""

    def __init__(self, ops, rt, sig, bmax):
        self.ops, self.sig, self.bmax = ops, sig, bmax
        _, g = _gen(sig)
        n = bmax + 1
        cin, cout, phase, kind, mode = sig["cin"], sig["cout"], sig["phase"], sig["kind"], sig["mode"]
        if phase is not None:
            K = 4 * cin
            w = _randn((cin, cout, 4, 4), g, "f32", 1 / math.sqrt(K))
            wp = ops.pack_convT_weight(w, mode != rt.MODE_F32)
            lp = ops.cast_f16(wp)[phase[0] * 2 + phase[1]] if sig["lp"] else None
            wp = wp[phase[0] * 2 + phase[1]]
            self.OH, self.OW = sig["H"], sig["W"]
        else:
            k = {"3x3": 3, "1x1": 1, "3x3s2": 3, "4x4s2": 4}[kind]
            K = k * k * cin + (sig["x2"][2] if sig["x2"] else 0)
            w = _randn((cout, cin, k, k), g, "f32", 1 / math.sqrt(K))
            wp = ops.pack_conv_weight(w, mode != rt.MODE_F32 and cin % 4 == 0 and cin > 4 and cout % 16 == 0)
            lp = ops.cast_f16(wp) if sig["lp"] else None
            self.OH, self.OW = ops.out_size(kind, sig["H"]), ops.out_size(kind, sig["W"])
        self.w, self.wp = w, wp
        self.x = _periodic(_randn((P, sig["H"], sig["W"], sig["ldi"]), g, sig["in_dt"]), n)
        self.bias = _randn((cout,), g, "f32") if sig["bias"] else None
        self.x2 = self.w2 = None
        if sig["x2"]:
            ldi2, _, cin2 = sig["x2"]
            self.x2 = _periodic(_randn((P, self.OH, self.OW, ldi2), g, sig["in_dt"]), n)
            self.w2 = _randn((cout, cin2, 1, 1), g, "f32", 1 / math.sqrt(K))
            p2 = ops.pack_conv_weight(self.w2, False)
            lp = ops.cast_f16(torch.cat([wp.reshape(cout, -1), p2.reshape(cout, -1)], dim=1).contiguous())
        self.lp = lp
        self.temb = self.temb_row = None
        if sig["temb"]:
            _, ld, off, per = sig["temb"]
            rows = _randn((P, ld), g, "f32")
            self.temb = (_periodic(rows, n) if per else rows[:1].contiguous())[:, off:]   # the engine's table view
            self.temb_row = rows[:1]
        self.res = None
        if sig["res"]:
            rdt, ldr, _ = sig["res"]
            self.res = _periodic(_randn((P, sig["OHf"], sig["OWf"], ldr), g, rdt), n)
        odt = torch.float16 if sig["out_dt"] == "f16" else torch.float32
        self.out = torch.empty((n, sig["OHf"], sig["OWf"], sig["ldo"]), device="cuda", dtype=odt)
        self.inputs = [t for t in (self.x, self.x2, self.res, self.wp, self.lp, self.bias, self.temb) if t is not None]
        self.pristine = [t.clone() for t in self.inputs]

    def kw(self, B, temb=None):
        """ops.conv keyword arguments at batch B; temb = (table, per_sample) replaces the layer's own rows."""
        s = self.sig
        kw = dict(mode=s["mode"], in_coff=s["in_coff"], cin=s["cin"], out_coff=s["out_coff"], act=s["act"],
                  phase=s["phase"], bias=self.bias, weight_lp=self.lp, out=self.out[:B])
        if self.x2 is not None:
            kw.update(x2=self.x2[:B], x2_coff=s["x2"][1], cin2=s["x2"][2])
        if s["temb"]:
            _, ld, _, per = s["temb"]
            t, per = temb if temb is not None else (self.temb[:B] if per else self.temb, per)
            kw.update(temb=t, temb_ld=ld, temb_per_sample=per)
        if self.res is not None:
            kw.update(residual=self.res[:B], res_coff=s["res"][2])
        return kw

    def route(self, B, **kw):
        return self.ops.conv_route(self.x[:B], self.wp, self.sig["kind"], self.sig["cout"], **self.kw(B, **kw))

    def window(self, t):
        s = self.sig
        step, (py, px) = (2, s["phase"]) if s["phase"] is not None else (1, (0, 0))
        return t[:, py::step, px::step, s["out_coff"]:s["out_coff"] + s["cout"]]

    def run(self, B, **kw):
        """Launch at batch B into a sentinel-filled buffer; returns the written window of samples 0..B-1."""
        fill_sentinel(self.out[:B + 1])
        self.ops.conv(self.x[:B], self.wp, self.sig["kind"], self.sig["cout"], **self.kw(B, **kw))
        torch.cuda.synchronize()
        return self.window(self.out[:B])

    def guard_violations(self, B):
        buf = self.out[:B + 1]
        return window_violations(buf, out_window(buf.shape, B, self.sig["phase"], self.sig["out_coff"],
                                                 self.sig["cout"], "cuda"))

    def inputs_changed(self):
        return not all(torch.equal(a, b) for a, b in zip(self.inputs, self.pristine))

    def reference(self, n):
        """float64 (ref, mag) of samples 0..n-1, computed on the GPU from the operand values the kernel reads."""
        s = self.sig
        step, (py, px) = (2, s["phase"]) if s["phase"] is not None else (1, (0, 0))
        xs = self.x[:n][..., s["in_coff"]:s["in_coff"] + s["cin"]]
        x2s = self.x2[:n][..., s["x2"][1]:s["x2"][1] + s["x2"][2]] if self.x2 is not None else None
        tembs = None
        if self.temb is not None:
            tembs = (self.temb[:n] if s["temb"][3] else self.temb)[:, :s["cout"]]
        ress = None
        if self.res is not None:
            ress = self.res[:n][:, py::step, px::step, s["res"][2]:s["res"][2] + s["cout"]]
        return conv_reference(s["kind"], s["phase"], xs, self.w, x2s, self.w2, self.bias, tembs, ress, s["act"])

    def name(self):
        s = self.sig
        return (f"conv {s['kind'] or 'convT'}{s['phase'] or ''} {s['H']}x{s['W']} cin={s['cin']}@{s['in_coff']}/"
                f"{s['ldi']} cout={s['cout']}@{s['out_coff']}/{s['ldo']} in={s['in_dt']} out={s['out_dt']} "
                f"res={s['res']} temb={s['temb']} act={s['act']} x2={s['x2']}")

    def in_bytes(self):
        """Per-sample bytes of the inputs an im2col route loads through an im2col descriptor."""
        s = self.sig
        elt = 2 if s["in_dt"] == "f16" else 4
        out = [s["H"] * s["W"] * s["ldi"] * elt]
        if s["x2"]:
            out.append(self.OH * self.OW * s["x2"][0] * elt)
        return out


def _tau_check(layer, route, ref, mag, j, e, got):
    """(ratio, within) of one element of sample j % P of the canonical reference."""
    tau = TAU["conv_tc" if route["path"] == 2 else "conv_cuda"]
    s = layer.sig
    r, _, _ = compare(got.reshape(1, 1, 1), ref[j][e].reshape(1, 1, 1), mag[j][e].reshape(1, 1, 1), tau, s["act"],
                      s["out_dt"] == "f16")
    return r


def _check_canonical(layer, rep):
    """Run at B = P and check every element against float64; returns (canonical window, ref, mag, route)."""
    route = layer.route(P)
    got = layer.run(P).clone()
    ref, mag = layer.reference(P)
    tau_key = "conv_tc" if route["path"] == 2 else "conv_cuda"
    worst = (0.0, None, None)
    for j in range(P):
        r, e, _ = compare(got[j], ref[j], mag[j], TAU[tau_key], layer.sig["act"], layer.sig["out_dt"] == "f16")
        if r > worst[0]:
            worst = (r, j, e)
    if worst[0] > 1:
        rep.fail(f"{layer.name()} B={P} [{conv_label(layer.sig, route)}]: sample {worst[1]} (y, x, channel) "
                 f"{worst[2]} ratio {worst[0]:.3g} against float64")
    return got, ref, mag, route, worst[0]


def _describe(layer, got, canon, ref, mag, route, b, e):
    j = b % P
    g, c = got[b][e], canon[j][e]
    r = _tau_check(layer, route, ref, mag, j, e, g)
    return (f"sample {b} (y, x, channel) {e}: got {float(g)!r}, canonical sample {j} holds {float(c)!r}; the got value "
            f"is {'within' if r <= 1 else 'OUTSIDE'} tau of float64 (ratio {r:.3g})")


class Report:
    def __init__(self):
        self.failures, self.fam = [], {}

    def fail(self, msg):
        self.failures.append(msg)

    def family(self, name):
        return self.fam.setdefault(name, dict(shapes=0, classes=0, replays=0, worst=0.0, secs=0.0))

    def print(self, title):
        print(f"\n{title}: family | shapes | distinct route classes | batch sizes replayed | worst ratio | wall s")
        for k, f in sorted(self.fam.items()):
            print(f"  {k:28s} {f['shapes']:5d} {f['classes']:6d} {f['replays']:7d} {f['worst']:9.4f} {f['secs']:8.1f}")

    def check(self):
        assert not self.failures, f"{len(self.failures)} failure(s):\n" + "\n".join(self.failures[:30])


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_conv_routes_are_batch_invariant(layers):
    ops, rt, convs, _ = layers
    rep = Report()
    classes = {}                                  # route label -> batch sizes replayed
    sides = {k: set() for k in ("halo", "bn", "ctas_per_sm", "bres", "second_round", "im2col_small")}
    for sig, bmax, prod in convs.values():
        t0 = time.perf_counter()
        layer = ConvLayer(ops, rt, sig, bmax)
        n0 = rt.launch_count()
        routes = [layer.route(B) for B in range(1, bmax + 1)]
        assert rt.launch_count() == n0, "the route sweep launched a kernel"
        picks = pick_batches(routes, layer.in_bytes(), {P} | prod)
        canon, ref, mag, croute, worst = _check_canonical(layer, rep)
        fam = rep.family(f"conv {ops.PATH_NAMES[routes[0]['path']]}")
        fam["shapes"] += 1
        fam["classes"] += len({route_class(r) for r in routes})
        fam["worst"] = max(fam["worst"], worst)
        widest = next((bn for bn in (256, 192, 128, 96, 64, 48, 32, 16) if sig["cout"] % bn == 0), None)
        for B in picks:
            want = routes[B - 1]
            head = (f"{layer.name()} B={B} [{conv_label(sig, want)} grid={want['grid']} ntiles={want['ntiles']}] "
                    f"against canonical B={P} [{conv_label(sig, croute)}]")
            got_route = layer.route(B)
            if got_route != want:
                rep.fail(f"{head}: replay route {got_route} != swept {want}")
            got = layer.run(B)
            bad = layer.guard_violations(B)
            if bad:
                rep.fail(f"{head}: bytes outside the output window changed at (sample, y, x, channel) {bad}")
            if layer.inputs_changed():
                rep.fail(f"{head}: an input buffer changed")
            mis = periodic_mismatch(got, canon)
            if mis is not None:
                rep.fail(f"{head}: {_describe(layer, got, canon, ref, mag, croute, *mis)}")
            fam["replays"] += 1
            classes.setdefault(conv_label(sig, want), set()).add(B)
            if want["path"] == 2:
                sides["halo"].add(want["halo"])
                if not want["halo"]:
                    sides["bn"].add("widest" if want["bn"] == widest else "narrowed")
                sides["ctas_per_sm"].add(want["ctas_per_sm"])
                sides["bres"].add(want["bres"])
                sides["second_round"].add(_second_round(want))
                if _im2col(want):
                    sides["im2col_small"].add(B * layer.in_bytes()[0] < IM2COL_SMALL)
        del layer, routes, canon, ref, mag
        torch.cuda.empty_cache()
        fam["secs"] += time.perf_counter() - t0
    print("\nroute classes replayed: route | batch sizes")
    for label, bs in sorted(classes.items()):
        print(f"  {label:78s} {len(bs):5d}")
    rep.print("convolutions across batch sizes")
    print(f"  sides reached: {dict((k, sorted(v, key=str)) for k, v in sides.items())}")
    assert rt.lib().cnb_tc_error_flag() == 0
    rep.check()
    assert sides["halo"] == {0, 1}, "halo and im2col"
    assert sides["bn"] == {"widest", "narrowed"}, "narrowed and widest BN"
    assert sides["ctas_per_sm"] == {1, 2}, "1 and 2 CTAs per SM"
    assert sides["bres"] == {0, 1}, "streamed and resident weights"
    assert sides["second_round"] == {False, True}, "ntiles <= grid and ntiles > grid"
    assert sides["im2col_small"] == {False, True}, "im2col inputs under and over 128 KiB"


@pytest.mark.gpu
def test_shared_and_per_sample_time_embedding_agree(layers):
    """One time-embedding row shared by the batch and B identical per-sample rows must give the same bits: a student
    called with a scalar sigma gets the shared row at B = 1 and per-sample rows at B > 1."""
    ops, rt, convs, _ = layers
    rep = Report()
    n = 0
    for sig, bmax, _ in convs.values():
        if not sig["temb"]:
            continue
        layer = ConvLayer(ops, rt, sig, bmax)
        off = sig["temb"][2]
        for B in sorted({1, P, bmax}):
            one = (layer.temb_row[:, off:], False)
            rows = (layer.temb_row.expand(B, -1).contiguous()[:, off:], True)     # same row stride as the table
            shared = layer.run(B, temb=one).clone()
            per = layer.run(B, temb=rows)
            n += 1
            mis = periodic_mismatch(per, shared)
            if mis is not None:
                b, e = mis
                rs, rp = layer.route(B, temb=one), layer.route(B, temb=rows)
                rep.fail(f"{layer.name()} B={B}: shared row [{conv_label(sig, rs)}] against per-sample rows "
                         f"[{conv_label(sig, rp)}]: sample {b} (y, x, channel) {e}: {float(shared[b][e])!r} against "
                         f"{float(per[b][e])!r}")
        del layer
        torch.cuda.empty_cache()
    print(f"\nshared against per-sample time embedding: {n} comparisons")
    assert n > 0
    assert rt.lib().cnb_tc_error_flag() == 0
    rep.check()


@pytest.mark.gpu
def test_split_groupnorm_is_batch_invariant(layers):
    """Split-statistics GroupNorm (the VAE decoder levels) at every B up to 256 and at the production batches and
    their shards: the number of row ranges per sample follows B, the statistics of a sample must not."""
    ops, rt, _, gns = layers
    rep = Report()
    fam = rep.family("groupnorm split-stats")
    for sig, bmax, prod in gns.values():
        H, W, C, G = sig["H"], sig["W"], sig["C"], sig["G"]
        if rt.lib().cnb_groupnorm_workspace_bytes(1, H * W, C, G, 1 if sig["in_dt"] == "f16" else 0) == 0:
            continue
        t0 = time.perf_counter()
        _, g = _gen(sig)
        means = torch.rand((C,), generator=g, device="cuda") * 12 - 6
        pool = torch.randn((P, H, W, C), generator=g, device="cuda") * 1.5 + means
        x = _periodic(pool.half() if sig["in_dt"] == "f16" else pool, bmax + 1)
        gamma = 1 + 0.5 * torch.randn((C,), generator=g, device="cuda")
        beta = 0.5 * torch.randn((C,), generator=g, device="cuda")
        x0 = x.clone()
        name = f"groupnorm {H}x{W} C={C} G={G} silu={sig['silu']} in={sig['in_dt']} out_f16={sig['out_f16']}"

        def run(B):
            return ops.groupnorm(x[:B], gamma, beta, G, sig["silu"], eps=sig["eps"], out_f16=sig["out_f16"])

        canon = run(P)
        ref, mag = groupnorm_reference(x[:P], gamma, beta, G, sig["eps"], sig["silu"])
        for j in range(P):
            r, e, _ = compare(canon[j], ref[j], mag[j], TAU["groupnorm"], sig["silu"], sig["out_f16"])
            fam["worst"] = max(fam["worst"], r)
            if r > 1:
                rep.fail(f"{name} B={P}: sample {j} (y, x, channel) {e} ratio {r:.3g} against float64")
        batches = sorted(set(range(1, min(bmax, 256) + 1)) | prod | {bmax})
        for B in batches:
            mis = periodic_mismatch(run(B), canon)
            if mis is not None:
                rep.fail(f"{name} B={B} against canonical B={P}: sample {mis[0]} (y, x, channel) {mis[1]} differs")
        if not torch.equal(x, x0):
            rep.fail(f"{name}: the input changed")
        fam["shapes"] += 1
        fam["replays"] += len(batches)
        del x, x0, canon, ref, mag
        torch.cuda.empty_cache()
        fam["secs"] += time.perf_counter() - t0
    rep.print("split-statistics GroupNorm across batch sizes")
    assert fam["shapes"] > 0, "no split-statistics GroupNorm shape in the workloads"
    rep.check()


# ---------------------------------------------------------------------------------------------------------------------
# CPU self-checks
# ---------------------------------------------------------------------------------------------------------------------
def _route(halo=0, bn=128, ctas=1, bres=0, grid=148, ntiles=1, path=2, epi=6):
    return dict(path=path, rb=128, bn=bn, epi=epi, halo=halo, bres=bres, ctas_per_sm=ctas, epi_alt=0, epi_nbuf=3,
                grid=grid, ntiles=ntiles, tiles_n=1, halo_r=0, tiles_y=0)


def test_pick_batches_covers_every_class_change():
    # B = 1..40: narrowed BN up to 9, widest BN with one CTA per SM up to 24, two CTAs per SM from 25, halo from 33;
    # a grid of 8 tiles with 3 tiles per sample: a second round from B = 3, a lone last tile at B = 3 (9 % 8 == 1)
    sms = 8
    routes = []
    for B in range(1, 41):
        nt = 3 * B
        if B <= 9:
            routes.append(_route(bn=64, grid=min(nt, sms), ntiles=nt))
        elif B <= 24:
            routes.append(_route(bn=128, grid=min(nt, sms), ntiles=nt))
        elif B <= 32:
            routes.append(_route(bn=128, ctas=2, bres=1, grid=min(nt, 2 * sms), ntiles=nt))
        else:
            routes.append(_route(halo=1, bres=1, epi=5, grid=min(nt, sms), ntiles=nt))
    picks = pick_batches(routes, in_bytes=[131072 // 6], extra=[16, 64])
    for b in (1, 9, 10, 24, 25, 32, 33, 40, 16):
        assert b in picks, b
    assert 3 in picks                         # first second round and first lone last tile of the first run
    assert 64 not in picks                    # above Bmax
    # the byte boundary: 6 samples are under 128 KiB, 7 are not
    assert 6 in picks and 7 in picks
    # the first second round of the two-CTA run: 3 * 25 = 75 tiles on 16 CTAs
    assert 25 in picks
    # a lone tile in the last round: 3 * B % 8 == 1 first at B = 11 (widest BN) and 35 (halo), 3 * B % 16 == 1 at 27
    assert {11, 27, 35} <= set(picks)
    # nothing else is picked inside a run
    assert picks == [1, 3, 6, 7, 9, 10, 11, 16, 24, 25, 27, 32, 33, 35, 40]


def test_pick_batches_byte_boundary_only_for_im2col():
    routes = [_route(halo=1, grid=B, ntiles=B) for B in range(1, 21)]
    assert pick_batches(routes, in_bytes=[131072 // 4]) == [1, 20]
    routes = [_route(path=1, grid=0, ntiles=0) for _ in range(10)]
    assert pick_batches(routes, extra=[4]) == [1, 4, 10]


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_periodic_comparator_flags_one_bit_and_a_shifted_sample(dtype):
    g = torch.Generator().manual_seed(3)
    canon = torch.randn((P, 6, 6, 24), generator=g).to(dtype)
    for B in (1, 7, 13):
        got = _periodic(canon, B)
        assert periodic_mismatch(got, canon) is None
        assert periodic_mismatch(got[..., 3:19], canon[..., 3:19]) is None     # a channel window view
        bad = got.clone()
        _bits(bad)[B - 1, 5, 4, 23] ^= 1                                     # the last bit of one element
        assert periodic_mismatch(bad, canon) == (B - 1, (5, 4, 23))
        if B > 1:
            shifted = got.clone()
            shifted[B - 1] = got[B - 2]                                      # a tile read the neighbouring sample
            assert periodic_mismatch(shifted, canon)[0] == B - 1
    neg0 = _periodic(torch.zeros((P, 2), dtype=dtype), 3)
    neg0[1, 1] = -0.0                                                        # equal as a number, not as bits
    assert periodic_mismatch(neg0, torch.zeros((P, 2), dtype=dtype)) == (1, (1,))
