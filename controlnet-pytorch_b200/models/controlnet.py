"""Drop-in for the reference's models/controlnet.py (DDPM ControlNet): frozen `trained_unet`, encoder-only
`control_copy_unet`, 4-conv hint block and zero convolutions, with the reference's constructor, checkpoint
splitting (controlnet.py:27-65,110-138), get_params (:140-156), forward(x, t, hint) (:158-225) and state_dict keys
(`trained_unet.*`, `control_copy_unet.*`, `control_copy_unet_hint_block.*`, `control_copy_unet_{down,mid}_zero_convs.*`).
"""
import torch
import torch.nn as nn

from . import _engine as E
from ._entry import host_entry
from ._controlnet_common import controlnet_forward, split_prefix
from .unet_base import Unet, get_time_embedding  # noqa: F401


def make_zero_module(module):
    return E.zero_(module)


class ControlNet(nn.Module):
    _AUX = ("control_copy_unet_hint_block.", "control_copy_unet_down_zero_convs.", "control_copy_unet_mid_zero_convs.")

    def __init__(self, model_config, model_locked=True, model_ckpt=None, device=None):
        super().__init__()
        self.model_locked = model_locked
        load = model_ckpt is not None and device is not None   # both are required (controlnet.py:27)
        ckpt = torch.load(model_ckpt, map_location=device) if load else None

        self.trained_unet = Unet(model_config)
        if load:
            print('Loading Trained Diffusion Model')
            full = 'trained_unet.conv_in.weight' in ckpt
            self.trained_unet.load_state_dict(split_prefix(ckpt, 'trained_unet.') if full else ckpt, strict=True)

        self.control_copy_unet = Unet(model_config, use_up=False)
        if load:
            print('Loading Control Diffusion Model')
            full = 'control_copy_unet.conv_in.weight' in ckpt
            self.control_copy_unet.load_state_dict(
                split_prefix(ckpt, 'control_copy_unet.', self._AUX) if full else ckpt, strict=False)

        c0 = self.trained_unet.down_channels[0]
        self.control_copy_unet_hint_block = nn.Sequential(
            nn.Conv2d(model_config['hint_channels'], 64, kernel_size=3, padding=(1, 1)), nn.SiLU(),
            nn.Conv2d(64, 128, kernel_size=3, padding=(1, 1)), nn.SiLU(),
            nn.Conv2d(128, c0, kernel_size=3, padding=(1, 1)), nn.SiLU(),
            make_zero_module(nn.Conv2d(c0, c0, kernel_size=1, padding=0)))
        dc, mc = self.trained_unet.down_channels, self.trained_unet.mid_channels
        self.control_copy_unet_down_zero_convs = nn.ModuleList(
            [make_zero_module(nn.Conv2d(dc[i], dc[i], kernel_size=1, padding=0)) for i in range(len(dc) - 1)])
        self.control_copy_unet_mid_zero_convs = nn.ModuleList(
            [make_zero_module(nn.Conv2d(mc[i], mc[i], kernel_size=1, padding=0)) for i in range(1, len(mc))])

        if load:   # a full ControlNet checkpoint also carries the hint block and the zero convolutions
            for attr, prefix in zip(("control_copy_unet_hint_block", "control_copy_unet_down_zero_convs",
                                     "control_copy_unet_mid_zero_convs"), self._AUX):
                sub = split_prefix(ckpt, prefix)
                if sub:
                    getattr(self, attr).load_state_dict(sub, strict=True)
        self._hint_cache = E.HintCache()

    def get_params(self):
        params = list(self.control_copy_unet.parameters())
        params += list(self.control_copy_unet_hint_block.parameters())
        params += list(self.control_copy_unet_down_zero_convs.parameters())
        params += list(self.control_copy_unet_mid_zero_convs.parameters())
        if not self.model_locked:
            params += list(self.trained_unet.ups.parameters())
            params += list(self.trained_unet.norm_out.parameters())
            params += list(self.trained_unet.conv_out.parameters())
        return params

    def _hint_feat(self, hint, mode):
        from .. import ops
        seq = self.control_copy_unet_hint_block
        return self._hint_cache.get(hint, list(seq.parameters()), mode,
                                    lambda: E.hint_stack_ddpm(seq, ops.nchw_to_nhwc(hint), mode))

    @host_entry
    def forward(self, x, t, hint):
        """eps = ControlNet(x_t, t, hint); x (B,C,H,W), hint (B,hint_channels,H,W) fp32 CUDA; t int (1,) or (B,)."""
        return controlnet_forward(self.trained_unet, self.control_copy_unet, self.control_copy_unet_down_zero_convs,
                                  self.control_copy_unet_mid_zero_convs, self._hint_feat, x, t, hint)

    def _forward_controlled(self, x, t, hint, scale=1.0, guidance=None):
        """forward with a conditioning scale on the down / mid zero convolutions and, with guidance = w, hint guidance
        eps = eu + w * (ec - eu) against the frozen U-Net (_controlnet_common.controlnet_forward).  Device tensors."""
        return controlnet_forward(self.trained_unet, self.control_copy_unet, self.control_copy_unet_down_zero_convs,
                                  self.control_copy_unet_mid_zero_convs, self._hint_feat, x, t, hint, scale=scale,
                                  guidance=guidance)
