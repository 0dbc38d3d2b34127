"""ControlNet wiring shared by the DDPM (models/controlnet.py:158-225) and LDM (models/controlnet_ldm.py:117-179)
variants, scheduled channels-last on libcnb200 kernels.

Dataflow (names as in the reference):
    a  = trained.conv_in(x)                     ; T_skips = inputs of trained.downs
    c  = control.conv_in(x) + hint_block(hint)  (hint feature cached: it depends on neither t nor x)
    C_skips[i] = zero_conv_i(c) written straight into the second half of the i-th up-block concat buffer,
                 with the trained skip added in the conv epilogue (controlnet.py:190-192, 216-218)
    mids: c = control.mid(c); a = trained.mid(a) + mid_zero_conv(c)   (injection fused in the epilogue, :207)
    ups on the trained U-Net, then norm_out / SiLU / conv_out.
"""
from .. import ops
from .. import runtime as rt
from . import _engine as E


def split_prefix(state, prefix, exclude=()):
    """{k[len(prefix):]: v} for the keys under `prefix` that are not under any of `exclude`."""
    return {k[len(prefix):]: v for k, v in state.items()
            if k.startswith(prefix) and not any(k.startswith(e) for e in exclude)}


_side_stream = E.side_stream


def controlnet_forward(trained, control, down_zero, mid_zero, hint_feat_fn, x, t, hint):
    import torch
    x = E._check_x(x)
    hint = E._check_x(hint)
    mode = rt.get_mode()
    dev = x.device
    xn = ops.nchw_to_nhwc(x)
    t = E.check_t(t, x.shape[0], dev)
    hf = hint_feat_fn(hint, mode)
    nmid = len(control.mids)

    def skip_sums(cs, t_skips):
        """zero_conv_i(control skip) + trained skip, written into the second half of the decoder's concat buffers
        (controlnet.py:190-192, 216-218)."""
        cats = []
        for i, c in enumerate(cs):
            B, H, W, C = c.shape
            zc = down_zero[i]
            cat = ops.empty(B, H, W, 2 * C, device=dev, dtype=c.dtype)
            E.conv16(c, zc.weight, "1x1", C, mode, bias=E.raw(zc.bias), residual=t_skips[i], out=cat, out_coff=C)
            cats.append(cat)
        return cats

    def inject(i, a, cm):
        """a + mid_zero_conv_i(control mid output): the sum rides in the zero conv's epilogue (:207)."""
        zc = mid_zero[i]
        return E.conv16(cm, zc.weight, "1x1", zc.out_channels, mode, bias=E.raw(zc.bias), residual=a)

    # The dependency graph of the reference's forward is wider than its statement order: the frozen encoder AND
    # trained.mids[0] never read a control tensor; trained.mids[i] needs control.mids[i-1] only through mid zero conv
    # i-1; the skip sums need the two encoders but nothing needs them before the decoder.  Under CUDA-graph capture the
    # forward is therefore laid out on four streams (forked / joined with events = parallel graph branches):
    #     cur  : trained conv_in -> downs -> mids[0] -> wait(control mid 0) inject -> mids[1] -> wait(...) inject -> ups
    #     side : control conv_in + hint feature -> downs -> mids[0] -> mids[1]
    #     skip : trained t-embedding rows; later wait(both encoders) -> the skip sums
    #     aux  : control t-embedding rows
    # The critical path loses one mid block per mid level, the skip sums and the t-embedding launches (measured, MNIST:
    # step at 128 samples 2.42 -> 2.24 ms, at 1024 samples 11.98 -> 11.80 ms; CelebHQ LDM at 256: 28.25 -> 27.7 ms; DESIGN.md 5);
    # the kernels of one branch fill the pipes the other leaves idle (MUFU-bound attention next to tensor- / HBM-bound
    # convolutions and GroupNorms).  Same kernels, same inputs, same order per tensor: results are bit-identical to the
    # sequential schedule.
    # Only under graph capture: in eager mode the extra stream bookkeeping (event waits, record_stream on every
    # hand-over tensor) is host time, which is what a small-batch eager loop is bound by (CelebHQ B = 16: 6.9 -> 19.7 ms).
    if not E.capture_parallel():
        plan_t = E.temb_plan(trained, E.unet_time(trained, t, dev))
        plan_c = E.temb_plan(control, E.unet_time(control, t, dev), with_ups=False)
        a = E.conv_in(trained, xn, mode)
        t_skips = []
        for d in trained.downs:
            t_skips.append(a)
            a = E.run_down(d, a, plan_t[d], mode)
        c = E.conv_in(control, xn, mode, residual=hf)
        cs = []
        for d in control.downs:
            cs.append(c)
            c = E.run_down(d, c, plan_c[d], mode)
        cms = []
        for mblk in control.mids:
            c = E.run_mid(mblk, c, plan_c[mblk], mode)
            cms.append(c)
        cats = skip_sums(cs, t_skips)
        for i in range(nmid):
            a = inject(i, E.run_mid(trained.mids[i], a, plan_t[trained.mids[i]], mode), cms[i])
    else:
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev, 0)
        skip = _side_stream(dev, 1)
        aux = _side_stream(dev, 2)
        E.prewarm_conv_in(trained, xn, mode)       # the padded fp16 copy both conv_in layers read: before the fork
        # the two t-embedding chains (4 small launches each) leave the critical paths as well: they are only needed by
        # the first resnet's conv1 epilogue, after conv_in and a GroupNorm
        skip.wait_stream(cur)
        aux.wait_stream(cur)
        with torch.cuda.stream(skip):
            plan_t = E.temb_plan(trained, E.unet_time(trained, t, dev))
            ev_pt = skip.record_event()
        with torch.cuda.stream(aux):
            plan_c = E.temb_plan(control, E.unet_time(control, t, dev), with_ups=False)
            ev_pc = aux.record_event()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            c = E.conv_in(control, xn, mode, residual=hf)
            side.wait_event(ev_pc)
            next(iter(plan_c.values())).table.record_stream(side)
            cs, cms, ev_mid = [], [], []
            for d in control.downs:
                cs.append(c)
                c = E.run_down(d, c, plan_c[d], mode)
            ev_enc = side.record_event()
            for mblk in control.mids:
                c = E.run_mid(mblk, c, plan_c[mblk], mode)
                cms.append(c)
                ev_mid.append(side.record_event())
        a = E.conv_in(trained, xn, mode)
        cur.wait_event(ev_pt)
        next(iter(plan_t.values())).table.record_stream(cur)
        t_skips = []
        for d in trained.downs:
            t_skips.append(a)
            a = E.run_down(d, a, plan_t[d], mode)
        skip.wait_stream(cur)                      # trained skips
        skip.wait_event(ev_enc)                    # control skips
        with torch.cuda.stream(skip):
            for tns in cs + t_skips:
                tns.record_stream(skip)
            cats = skip_sums(cs, t_skips)
        for i in range(nmid):
            a = E.run_mid(trained.mids[i], a, plan_t[trained.mids[i]], mode)
            cur.wait_event(ev_mid[i])
            cms[i].record_stream(cur)
            a = inject(i, a, cms[i])
        cur.wait_stream(side)
        cur.wait_stream(skip)
        cur.wait_stream(aux)
        for tns in cats:
            tns.record_stream(cur)

    for u in trained.ups:
        a = E.run_up(u, a, None, plan_t[u], mode, cat=cats.pop())
    return ops.nhwc_to_nchw(E.conv_out(trained, a, mode))
