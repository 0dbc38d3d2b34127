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
import contextlib

import torch

from .. import ops
from .. import runtime as rt
from . import _engine as E


def split_prefix(state, prefix, exclude=()):
    """{k[len(prefix):]: v} for the keys under `prefix` that are not under any of `exclude`."""
    return {k[len(prefix):]: v for k, v in state.items()
            if k.startswith(prefix) and not any(k.startswith(e) for e in exclude)}


_STREAMS = {}


class _Branches:
    """The parallel graph branches of one ControlNet forward.  Under CUDA-graph capture each named branch runs on a
    side stream of its own: it forks from one event recorded when this object is made, orders itself after other
    work only through `wait`, and `join` brings every branch back into the current stream.  Outside capture every
    method is a no-op and all work runs on the current stream in program order: the stream bookkeeping (event waits,
    record_stream on every hand-over tensor) is host time, which is what a small-batch eager loop is bound by
    (CelebHQ B = 16: 6.9 -> 19.7 ms)."""

    def __init__(self, dev):
        self.dev = dev
        self.capturing = torch.cuda.is_current_stream_capturing()
        if self.capturing:
            self.cur = torch.cuda.current_stream(dev)
            self.fork = self.cur.record_event()
            self.streams = {}

    def on(self, name):
        """Context in which work is enqueued on branch `name`."""
        if not self.capturing:
            return contextlib.nullcontext()
        s = self.streams.get(name)
        if s is None:
            key = (str(self.dev), self.cur.cuda_stream, name)
            if key not in _STREAMS:
                _STREAMS[key] = torch.cuda.Stream(device=self.dev)
            s = self.streams[name] = _STREAMS[key]
            s.wait_event(self.fork)
        return torch.cuda.stream(s)

    def record(self):
        """An event marking the work enqueued so far on the current stream."""
        return torch.cuda.current_stream(self.dev).record_event() if self.capturing else None

    def wait(self, ev, *tensors):
        """The current stream waits for `ev` and then reads `tensors`, which another branch made."""
        if self.capturing:
            s = torch.cuda.current_stream(self.dev)
            s.wait_event(ev)
            for tns in tensors:
                tns.record_stream(s)

    def join(self, *tensors):
        """The stream that made this object waits for every branch and then reads `tensors`."""
        if self.capturing:
            for s in self.streams.values():
                self.cur.wait_stream(s)
            for tns in tensors:
                tns.record_stream(self.cur)


def controlnet_forward(trained, control, down_zero, mid_zero, hint_feat_fn, x, t, hint):
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
    # i-1; the skip sums need the two encoders but nothing needs them before the decoder; the two t-embedding chains
    # (4 small launches each) are only needed by the first resnet's conv1 epilogue, after conv_in and a GroupNorm.
    # Outside capture the statements below run in their written order on one stream.  Under CUDA-graph capture each
    # one also runs on a branch (forked / joined with events = parallel graph branches):
    #     (current) : trained conv_in -> downs -> mids[0] -> wait(control mid 0) inject -> mids[1] -> ... -> ups
    #     side      : control conv_in + hint feature -> downs -> mids[0] -> mids[1]
    #     skip      : trained t-embedding rows; later wait(both encoders) -> the skip sums
    #     aux       : control t-embedding rows
    # The critical path loses one mid block per mid level, the skip sums and the t-embedding launches (measured, MNIST:
    # step at 128 samples 2.42 -> 2.24 ms, at 1024 samples 11.98 -> 11.80 ms; CelebHQ LDM at 256: 28.25 -> 27.7 ms; DESIGN.md 5);
    # the kernels of one branch fill the pipes the other leaves idle (MUFU-bound attention next to tensor- / HBM-bound
    # convolutions and GroupNorms).  Same kernels, same inputs, same order per tensor: results are bit-identical to the
    # eager (one-stream) run.
    E.prewarm_conv_in(trained, xn, mode)       # the padded fp16 copy both conv_in layers read: before the fork
    br = _Branches(dev)
    with br.on("skip"):
        plan_t = E.temb_plan(trained, E.unet_time(trained, t, dev))
        ev_pt = br.record()
    with br.on("aux"):
        plan_c = E.temb_plan(control, E.unet_time(control, t, dev), with_ups=False)
        ev_pc = br.record()
    a = E.conv_in(trained, xn, mode)
    br.wait(ev_pt, next(iter(plan_t.values())).table)
    t_skips = []
    for d in trained.downs:
        t_skips.append(a)
        a = E.run_down(d, a, plan_t[d], mode)
    ev_tenc = br.record()
    with br.on("side"):
        c = E.conv_in(control, xn, mode, residual=hf)
        br.wait(ev_pc, next(iter(plan_c.values())).table)
        cs, cms, ev_mid = [], [], []
        for d in control.downs:
            cs.append(c)
            c = E.run_down(d, c, plan_c[d], mode)
        ev_cenc = br.record()
        for mblk in control.mids:
            c = E.run_mid(mblk, c, plan_c[mblk], mode)
            cms.append(c)
            ev_mid.append(br.record())
    with br.on("skip"):
        br.wait(ev_tenc, *t_skips)
        br.wait(ev_cenc, *cs)
        cats = skip_sums(cs, t_skips)
    for i in range(nmid):
        a = E.run_mid(trained.mids[i], a, plan_t[trained.mids[i]], mode)
        br.wait(ev_mid[i], cms[i])
        a = inject(i, a, cms[i])
    br.join(*cats)

    for u in trained.ups:
        a = E.run_up(u, a, None, plan_t[u], mode, cat=cats.pop())
    return ops.nhwc_to_nchw(E.conv_out(trained, a, mode))
