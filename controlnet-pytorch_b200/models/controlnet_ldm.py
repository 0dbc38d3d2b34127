"""Drop-in for the reference's models/controlnet_ldm.py (LDM ControlNet on VAE latents): same wiring as the DDPM
variant on unet_cond_base.Unet; the hint block is the stride-2 pyramid from `canny_im_size` down to the latent size
(controlnet_ldm.py:45-79) and the attribute prefixes are `control_unet*` (:36,:79,:82,:91).
"""
import torch
import torch.nn as nn

from .. import ops
from . import _engine as E
from ._entry import host_entry
from ._controlnet_common import controlnet_forward
from .blocks import get_time_embedding  # noqa: F401
from .unet_cond_base import Unet


def make_zero_module(module):
    return E.zero_(module)


class ControlNet(nn.Module):
    def __init__(self, im_channels, model_config, model_locked=True, model_ckpt=None, device=None,
                 down_sample_factor=32):
        super().__init__()
        self.model_locked = model_locked
        load = model_ckpt is not None and device is not None
        self.trained_unet = Unet(im_channels, model_config)
        if load:
            print('Loading Trained Diffusion Model')
            self.trained_unet.load_state_dict(torch.load(model_ckpt, map_location=device), strict=True)
        self.control_unet = Unet(im_channels, model_config, use_up=False)
        if load:
            print('Loading Control Diffusion Model')
            self.control_unet.load_state_dict(torch.load(model_ckpt, map_location=device), strict=False)

        ch, factor = 16, down_sample_factor
        stages = [nn.Sequential(nn.Conv2d(model_config['hint_channels'], ch, kernel_size=3, padding=(1, 1)), nn.SiLU())]
        while factor > 1:
            stages.append(nn.Sequential(nn.Conv2d(ch, ch * 2, kernel_size=3, padding=(1, 1), stride=2), nn.SiLU(),
                                        nn.Conv2d(ch * 2, ch * 2, kernel_size=3, padding=(1, 1))))
            ch, factor = ch * 2, factor / 2
        c0 = self.trained_unet.down_channels[0]
        stages.append(nn.Sequential(nn.Conv2d(ch, c0, kernel_size=3, padding=(1, 1)), nn.SiLU(),
                                    make_zero_module(nn.Conv2d(c0, c0, kernel_size=1, padding=0))))
        self.control_unet_hint_block = nn.Sequential(*stages)

        dc, mc = self.trained_unet.down_channels, self.trained_unet.mid_channels
        self.control_unet_down_zero_convs = nn.ModuleList(
            [make_zero_module(nn.Conv2d(dc[i], dc[i], kernel_size=1, padding=0)) for i in range(len(dc) - 1)])
        self.control_unet_mid_zero_convs = nn.ModuleList(
            [make_zero_module(nn.Conv2d(mc[i], mc[i], kernel_size=1, padding=0)) for i in range(1, len(mc))])
        self._hint_cache = E.HintCache()

    def get_params(self):
        params = list(self.control_unet.parameters())
        params += list(self.control_unet_hint_block.parameters())
        params += list(self.control_unet_down_zero_convs.parameters())
        params += list(self.control_unet_mid_zero_convs.parameters())
        if not self.model_locked:
            params += list(self.trained_unet.ups.parameters())
            params += list(self.trained_unet.norm_out.parameters())
            params += list(self.trained_unet.conv_out.parameters())
        return params

    def _pyramid(self, hint_nhwc, mode):
        """3x3+SiLU | [3x3 s2 + SiLU, 3x3] per halving | 3x3+SiLU, 1x1  (controlnet_ldm.py:45-79)."""
        stages = list(self.control_unet_hint_block)

        def cv(conv, h, kind, act):
            return E.conv16(h, conv.weight, kind, conv.out_channels, mode, bias=E.raw(conv.bias), act=act)
        h = cv(stages[0][0], hint_nhwc, "3x3", 1)
        for st in stages[1:-1]:
            h = cv(st[0], h, "3x3s2", 1)
            h = cv(st[2], h, "3x3", 0)
        h = cv(stages[-1][0], h, "3x3", 1)
        return cv(stages[-1][2], h, "1x1", 0)

    def _hint_feat(self, hint, mode):
        seq = self.control_unet_hint_block
        return self._hint_cache.get(hint, list(seq.parameters()), mode,
                                    lambda: self._pyramid(ops.nchw_to_nhwc(hint), mode))

    @host_entry
    def forward(self, x, t, hint):
        return controlnet_forward(self.trained_unet, self.control_unet, self.control_unet_down_zero_convs,
                                  self.control_unet_mid_zero_convs, self._hint_feat, x, t, hint)

    def _forward_controlled(self, x, t, hint, scale=1.0, guidance=None):
        """forward with a conditioning scale on the down / mid zero convolutions and, with guidance = w, hint guidance
        eps = eu + w * (ec - eu) against the frozen U-Net (_controlnet_common.controlnet_forward).  Device tensors."""
        return controlnet_forward(self.trained_unet, self.control_unet, self.control_unet_down_zero_convs,
                                  self.control_unet_mid_zero_convs, self._hint_feat, x, t, hint, scale=scale,
                                  guidance=guidance)
