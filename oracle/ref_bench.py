"""BENCH / TEST INFRASTRUCTURE -- drives the reference's own implementation of the hot path for the baseline legs of
bench.py (never imported by the product path).

Two back ends, in order of preference:

* ``kind == "reference"``: the UNMODIFIED reference modules -- ``UNetModel`` (openaimodel.py:837-885), ``Decoder``
  (model.py:653-686), ``Generator`` (hifigan/models.py:149-165) driven by the reference ``DDIMSampler``
  (ddim.py:166-355, two ``apply_model`` calls per step as ddim.py:293-296) -- imported from ``$ALDM_REFERENCE_ROOT`` or
  from ``baseline/_ref`` (``pip install --no-deps --target baseline/_ref`` of the reference, git-ignored), with the package
  ``__init__`` files bypassed (oracle/ref_loader.py).  Only paths the caller names or inside the tree are searched.
* ``kind == "port"``: oracle/functional.py, the torch restatement pinned against those modules by the fixtures.

Both run the seeded synthetic checkpoint / conditioning of SURVEY.md 8d on the device they are given.
"""
from __future__ import annotations

import contextlib
import io
import os
import time
import types
from typing import Optional

import torch

from audioldm2_b200 import arch, synth
from . import functional as OF
from . import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _locate_reference() -> Optional[str]:
    for cand in (os.environ.get("ALDM_REFERENCE_ROOT"), os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isdir(os.path.join(cand, "audioldm2", "latent_diffusion")):
            return cand
    return None


class _Stub:
    """The attributes DDIMSampler touches on ``self.model`` (SURVEY.md 8c)."""

    def __init__(self, unet, tables, device):
        self.unet, self.device = unet, device
        self.num_timesteps, self.parameterization = 1000, "eps"
        for k, v in tables.items():
            setattr(self, k, v.to(device))

    def apply_model(self, x, t, c):              # DiffusionWrapper.forward -> UNetModel.forward (ddpm.py:1875-1878)
        return self.unet(x, t, y=c["y"], context_list=c["context_list"], context_attn_mask_list=c["mask_list"])

    def q_sample(self, x_start, t, noise=None):  # ddpm.py:430-436
        noise = torch.randn_like(x_start) if noise is None else noise
        a = self.sqrt_alphas_cumprod[t].reshape(-1, 1, 1, 1)
        b = self.sqrt_one_minus_alphas_cumprod[t].reshape(-1, 1, 1, 1)
        return a * x_start + b * noise


class ReferencePath:
    """x_T -> S x (2 UNet calls, CFG, DDIM update) -> VAE decode -> HiFi-GAN on ``device`` with the reference's code."""

    def __init__(self, model_name: str, batch: int, device, t5_len: int = 32, cond_seed: int = 77, force_port: bool = False):
        self.cfg = cfg = arch.model_config(model_name)
        self.B, self.dev = batch, torch.device(device)
        self.tables = OF.ddpm_tables(cfg["linear_start"], cfg["linear_end"], cfg["timesteps"])
        usd, vsd, hsd = synth.unet_state_dict(cfg["unet"]), synth.vae_state_dict(cfg["vae"]), synth.vocoder_state_dict(cfg["vocoder"])
        self.cond, self.unc = synth.conditioning(cfg, batch, seed=cond_seed, t5_len=t5_len, device=self.dev)
        root = None if force_port else _locate_reference()
        self.kind = "port"
        self.where = "oracle/functional.py (torch restatement of the reference modules)"
        if root is not None:
            try:
                ref_loader.REF_ROOT = root
                R = ref_loader.load()
                u = cfg["unet"]
                kw = dict(image_size=64, use_spatial_transformer=True)
                for k in ("in_channels", "out_channels", "model_channels", "attention_resolutions", "num_res_blocks", "channel_mult",
                          "num_head_channels", "transformer_depth", "context_dim", "extra_film_condition_dim"):
                    kw[k] = u[k]
                kw["context_dim"] = list(kw["context_dim"])
                self.unet = R.UNetModel(**kw).eval()
                self.unet.load_state_dict(usd, strict=True)
                v = cfg["vae"]
                self.dec = R.Decoder(double_z=True, z_channels=v["z_channels"], resolution=256, in_channels=v["in_channels"],
                                     out_ch=v["out_ch"], ch=v["ch"], ch_mult=list(v["ch_mult"]), num_res_blocks=v["num_res_blocks"],
                                     attn_resolutions=[], dropout=0.0).eval()
                self.dec.load_state_dict({k[len("decoder."):]: t for k, t in vsd.items() if k.startswith("decoder.")}, strict=True)
                self.voc = R.Generator(types.SimpleNamespace(**cfg["vocoder"])).eval()
                self.voc.remove_weight_norm()
                self.voc.load_state_dict(hsd, strict=True)
                for m in (self.unet, self.dec, self.voc):
                    m.to(self.dev)
                self.pq = (vsd["post_quant_conv.weight"].to(self.dev), vsd["post_quant_conv.bias"].to(self.dev))
                self.sampler = R.DDIMSampler(_Stub(self.unet, self.tables, self.dev), device=self.dev)
                self.kind = "reference"
                self.where = f"unmodified reference modules from {root} (UNetModel, Decoder, Generator, DDIMSampler)"
            except Exception as e:   # pragma: no cover
                self.where = f"oracle/functional.py (reference import failed: {e!r})"
        if self.kind == "port":
            mv = lambda sd: {k: t.to(self.dev) for k, t in sd.items()}
            self.usd, self.vsd, self.hsd = mv(usd), mv(vsd), mv(hsd)

    # ---- sampling ------------------------------------------------------------------------------------
    @torch.no_grad()
    def sample(self, S: int, n_steps: Optional[int] = None, guidance: float = 3.5, x_T=None):
        """The first ``n_steps`` (default all) of an S-step DDIM run, eta 1.0.  Noise: torch.randn on ``device`` in the
        reference's order (x_T at ddim.py:191, then one draw per step at ddim.py:351)."""
        cfg, B = self.cfg, self.B
        C_, T, F_ = cfg["latent"]
        if self.kind == "reference":
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                self.sampler.make_schedule(ddim_num_steps=S, ddim_eta=1.0, verbose=False)
                # ddim.py:199-207: `timesteps` keeps ddim_timesteps[:int(timesteps) - 1], i.e. the LOW-noise end of the
                # schedule (cost per step is identical); +1.5 keeps the float round trip inside int() exact
                ts = None if n_steps is None or n_steps >= S else n_steps + 1.5
                img, _ = self.sampler.ddim_sampling(self.cond, (B, C_, T, F_), x_T=x_T, timesteps=ts,
                                                    unconditional_guidance_scale=guidance, unconditional_conditioning=self.unc)
            return img
        img = torch.randn(B, C_, T, F_, device=self.dev) if x_T is None else x_T
        sched = OF.ddim_schedule(self.tables, S, 1.0)
        for st in sched[-(n_steps or S):]:          # same (low-noise) subset as the reference's `timesteps` argument
            ts = torch.full((B,), st["t"], dtype=torch.long, device=self.dev)
            e_u = OF.unet_forward(self.usd, cfg["unet"], img, ts, self.unc["context_list"], self.unc["mask_list"], self.unc["y"])
            e_c = OF.unet_forward(self.usd, cfg["unet"], img, ts, self.cond["context_list"], self.cond["mask_list"], self.cond["y"])
            img, _ = OF.ddim_update(img, e_u, e_c, torch.randn(B, C_, T, F_, device=self.dev), st, guidance)
        return img

    @torch.no_grad()
    def decode(self, z):
        """decode_first_stage + mel_spectrogram_to_waveform (ddpm.py:922-939), waveform left on the device."""
        if self.kind == "reference":
            h = torch.nn.functional.conv2d(z / 1.0, self.pq[0], self.pq[1])          # autoencoder.py:112
            mel = self.dec(h)
            return self.voc(mel.squeeze(1).permute(0, 2, 1))                        # ddpm.py:932-935
        mel = OF.vae_decode(self.vsd, self.cfg["vae"], z)
        return OF.vocoder_forward(self.hsd, self.cfg["vocoder"], mel.squeeze(1).permute(0, 2, 1))


def set_precision(mode: str):
    """'high' = the CLI's setting (bin/audioldm2:139 torch.set_float32_matmul_precision("high")) on top of torch's default
    cuDNN TF32 convolutions; 'default' = torch defaults (TF32 convolutions, fp32 matmuls); 'fp32' = no TF32 anywhere."""
    torch.backends.cudnn.allow_tf32 = mode != "fp32"
    torch.backends.cuda.matmul.allow_tf32 = mode == "high"


def time_cuda(ref: ReferencePath, S: int, n_steps: Optional[int], seed: int = 42):
    """CUDA-event timing of sampler + decode; returns (latent, wave, s_sampler, s_decode)."""
    torch.manual_seed(seed)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    e[0].record()
    z = ref.sample(S, n_steps)
    e[1].record()
    w = ref.decode(z)
    e[2].record()
    torch.cuda.synchronize()
    return z, w, e[0].elapsed_time(e[1]) * 1e-3, e[1].elapsed_time(e[2]) * 1e-3


def time_cpu(ref: ReferencePath, S: int, n_steps: int):
    t0 = time.perf_counter()
    z = ref.sample(S, n_steps)
    t1 = time.perf_counter()
    ref.decode(z)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1
