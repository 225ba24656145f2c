"""Drop-in for model_scripts/ddpm_3d_ldm/vae.py (reference file:line in docstrings).

Same classes, constructor signatures, attributes and state_dict keys.  `encode`,
`encode_to_latent`, `decode`, `decode_from_latent` and `forward` run the B200 engine
(vae_engine.VAE3DProgram): inference programs whenever no gradient is required -- latents for LDM
training (train.py:386-388, frozen VAE under no_grad), latent statistics (train.py:351-364),
decoding samples (show_model.py:255) -- and training programs (forward + backward launch lists
behind one autograd node each for the encoder and the decoder) for the VAE's own training stage
(train.py:258-300: `recon, mu, logvar = vae(x)`, L1 + KL loss, GradScaler, DDP).
"""
import torch
import torch.nn as nn

from ... import _lib
from ...modules import EngineModule, ProgramFunction, on_input_device
from ...split_engine import VAE3DSplitProgram
from ...vae_engine import VAE3DProgram


class ResidualBlock3DNoTime(nn.Module):
    """Parameter holder for ResidualBlock3DNoTime (vae.py:5-17)."""

    def __init__(self, in_channels, out_channels, groups=8):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, in_channels)
        self.act1 = nn.SiLU()
        self.conv1 = nn.Conv3d(in_channels, out_channels, 3, padding=1)
        self.norm2 = nn.GroupNorm(groups, out_channels)
        self.act2 = nn.SiLU()
        self.conv2 = nn.Conv3d(out_channels, out_channels, 3, padding=1)
        if in_channels != out_channels:
            self.skip = nn.Conv3d(in_channels, out_channels, 1)
        else:
            self.skip = nn.Identity()


class Encoder3D(nn.Module):
    """Parameter holder for Encoder3D (vae.py:25-47)."""

    def __init__(self, in_channels=4, base_channels=32, num_down=3, latent_channels=8, groups=8):
        super().__init__()
        self.num_down = num_down
        self.in_conv = nn.Conv3d(in_channels, base_channels, 3, padding=1)
        downs = []
        cur_ch = base_channels
        for i in range(num_down):
            downs.append(ResidualBlock3DNoTime(cur_ch, cur_ch, groups))
            if i != num_down - 1:
                downs.append(ResidualBlock3DNoTime(cur_ch, cur_ch * 2, groups))
                downs.append(nn.Conv3d(cur_ch * 2, cur_ch * 2, 4, stride=2, padding=1))
                cur_ch *= 2
        self.downs = nn.ModuleList(downs)
        self.out_channels = cur_ch
        self.to_mu_logvar = nn.Conv3d(cur_ch, 2 * latent_channels, 3, padding=1)


class Decoder3D(nn.Module):
    """Parameter holder for Decoder3D (vae.py:58-81)."""

    def __init__(self, out_channels=4, base_channels=32, num_down=3, latent_channels=8,
                 enc_out_channels=None, groups=8):
        super().__init__()
        if enc_out_channels is None:
            enc_out_channels = base_channels * (2 ** (num_down - 1))
        cur_ch = enc_out_channels
        self.from_latent = nn.Conv3d(latent_channels, cur_ch, 3, padding=1)
        ups = []
        for i in reversed(range(num_down)):
            ups.append(ResidualBlock3DNoTime(cur_ch, cur_ch, groups))
            if i != 0:
                ups.append(ResidualBlock3DNoTime(cur_ch, cur_ch // 2, groups))
                ups.append(nn.ConvTranspose3d(cur_ch // 2, cur_ch // 2, 4, stride=2, padding=1))
                cur_ch //= 2
        self.ups = nn.ModuleList(ups)
        self.out_conv = nn.Conv3d(cur_ch, out_channels, 3, padding=1)


class VAE3D(EngineModule):
    """vae.py:90-127."""

    MAX_PROGRAMS = 6   # stage 1 alternates encoder / decoder training and inference programs
    # "bf16" (default) | "split": fp32-class parity with the reference's un-autocast decode
    # (show_model.py:255) on the bf16 kernels, see split_engine.py.  Inference only.
    precision = "bf16"

    def __init__(self, in_channels=4, base_channels=32, num_down=3, latent_channels=8, groups=8):
        super().__init__()
        self.encoder = Encoder3D(in_channels, base_channels, num_down, latent_channels, groups)
        self.decoder = Decoder3D(in_channels, base_channels, num_down, latent_channels,
                                 enc_out_channels=self.encoder.out_channels, groups=groups)

    # ------------------------------------------------------------------ engine plumbing
    def _program(self, mode: str, x: torch.Tensor, training: bool = False,
                 wgrad: bool = True) -> VAE3DProgram:
        """The cached engine program for (mode, shape).  training=True, wgrad=False: the training
        program without parameter gradients (decoder input gradients for guided sampling)."""
        self._check_input(x)
        if x.dim() != 5:
            raise _lib.MriError(f"VAE3D expects (B, C, D, H, W), got {tuple(x.shape)}")
        if self.precision == "split":
            if training:
                raise _lib.MriError("precision = 'split' is an inference mode (use 'bf16' for training)")
            skey = (mode, int(x.shape[0]), tuple(int(s) for s in x.shape[2:]), "split")
            return self.get_program(skey, lambda: VAE3DSplitProgram(self, mode, skey[1], skey[2]))
        if self.precision != "bf16":
            raise _lib.MriError(f"unknown precision {self.precision!r}: 'bf16' or 'split'")
        key = (mode, int(x.shape[0]), tuple(int(s) for s in x.shape[2:]), bool(training))
        if not wgrad:
            key += ("dgrad",)
        return self.get_program(key, lambda: VAE3DProgram(self, mode, key[1], key[2], training=key[3],
                                                          wgrad=wgrad))

    def _run(self, mode: str, x: torch.Tensor, part: nn.Module) -> torch.Tensor:
        xf = x.float().contiguous()
        needs = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in part.parameters()))
        if not needs:
            return self._program(mode, x).forward(xf).clone()
        if mode == "encode" and x.requires_grad:
            raise _lib.MriError("VAE3D.encode: a gradient w.r.t. the input volume is not provided (the "
                                "reference's training never asks for one, train.py:262-276)")
        # training (train.py:258-300): forward + backward launch lists behind one autograd node
        prog = self._program(mode, x, training=True)
        prog.param_list = list(part.parameters())
        return ProgramFunction.apply(prog, lambda: prog.forward(xf), xf if mode == "decode" else None,
                                     *prog.param_list)

    @on_input_device
    def encode(self, x):
        """vae.py:102-104: (mu, logvar), each (B, latent, D/4, H/4, W/4)."""
        cin = self.encoder.in_conv.weight.shape[1]
        if x.shape[1] != cin:
            raise _lib.MriError(f"expected {cin} input channels, got {x.shape[1]}")
        stats = self._run("encode", x, self.encoder)
        mu, logvar = torch.chunk(stats, 2, dim=1)
        return mu, logvar

    def reparameterize(self, mu, logvar):
        """vae.py:106-109."""
        std = torch.exp(0.5 * logvar)
        eps = torch.randn_like(std)
        return mu + eps * std

    @on_input_device
    def decode(self, z):
        """vae.py:111-112."""
        lat = self.decoder.from_latent.weight.shape[1]
        if z.shape[1] != lat:
            raise _lib.MriError(f"expected {lat} latent channels, got {z.shape[1]}")
        return self._run("decode", z, self.decoder)

    @on_input_device
    def forward(self, x):
        """vae.py:114-118."""
        mu, logvar = self.encode(x)
        z = self.reparameterize(mu, logvar)
        recon = self.decode(z)
        return recon, mu, logvar

    @torch.no_grad()
    @on_input_device
    def encode_to_latent(self, x):
        """vae.py:120-124: deterministic latent mean for diffusion."""
        mu, logvar = self.encode(x)
        return mu

    @torch.no_grad()
    @on_input_device
    def decode_from_latent(self, z):
        """vae.py:126-128."""
        return self.decode(z)
