"""Generate the golden fixtures by running the UNMODIFIED reference modules.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py [--only NAME] [--skip-200]

For every fixture the reference nn.Module is constructed from the same config dict the
reference uses, loaded (strict) with the seeded synthetic ``state_dict`` of
``audioldm2_b200.synth`` -- which also proves that ``audioldm2_b200.arch`` reproduces the
reference key names and shapes -- and run on CPU in fp32.  Inputs are regenerated from seeds
by ``tests/golden/cases.py`` so only the outputs are stored.
"""
from __future__ import annotations

import argparse
import ast
import json
import os
import sys
import time
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from audioldm2_b200 import arch, synth          # noqa: E402
from oracle import functional as OF             # noqa: E402
from oracle import ref_loader                   # noqa: E402
from tests.golden import cases                  # noqa: E402


def _save(name, d):
    path = os.path.join(HERE, name + ".pt")
    torch.save(cases.thin({k: (v.contiguous() if torch.is_tensor(v) else v) for k, v in d.items()}), path)
    print(f"wrote {path} ({os.path.getsize(path) / 1e3:.0f} KB)")


def ref_unet(R, ucfg):
    kw = dict(image_size=64, use_spatial_transformer=True)
    for k in ("in_channels", "out_channels", "model_channels", "attention_resolutions", "num_res_blocks",
              "channel_mult", "num_head_channels", "transformer_depth", "context_dim",
              "extra_film_condition_dim"):
        kw[k] = ucfg[k]
    kw["context_dim"] = list(kw["context_dim"])
    m = R.UNetModel(**kw).eval()
    m.load_state_dict(synth.unet_state_dict(ucfg), strict=True)
    return m


def ref_vae(R, vcfg):
    dd = dict(double_z=True, z_channels=vcfg["z_channels"], resolution=256, in_channels=vcfg["in_channels"],
              out_ch=vcfg["out_ch"], ch=vcfg["ch"], ch_mult=list(vcfg["ch_mult"]),
              num_res_blocks=vcfg["num_res_blocks"], attn_resolutions=[], dropout=0.0)
    dec, enc = R.Decoder(**dd).eval(), R.Encoder(**dd).eval()
    sd = synth.vae_state_dict(vcfg)
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")}, strict=True)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}, strict=True)
    return dec, enc, sd


def ref_vocoder(R, vcfg):
    h = types.SimpleNamespace(**vcfg)
    g = R.Generator(h).eval()
    g.remove_weight_norm()                      # utilities/model.py:139-140
    g.load_state_dict(synth.vocoder_state_dict(vcfg), strict=True)
    return g


@torch.no_grad()
def gen_unet(R, name, cfg, B, t5_len=32):
    m = ref_unet(R, cfg["unet"])
    x, t, cond, unc = cases.unet_inputs(cfg, B, t5_len=t5_len)
    out = {}
    for tag, c in (("cond", cond), ("uncond", unc)):
        t0 = time.time()
        out["eps_" + tag] = m(x, t, y=c["y"], context_list=c["context_list"], context_attn_mask_list=c["mask_list"])
        print(f"  {name}/{tag}: {time.time() - t0:.2f}s")
    _save(name, out)


@torch.no_grad()
def gen_vae(R, name, cfg, B):
    dec, enc, sd = ref_vae(R, cfg["vae"])
    z = cases.latent(cfg, B, seed=5)
    h = torch.nn.functional.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])   # autoencoder.py:112
    mel = dec(h)
    melin = cases.mel_input(cfg, B)
    mom = torch.nn.functional.conv2d(enc(melin), sd["quant_conv.weight"], sd["quant_conv.bias"])  # autoencoder.py:106-107
    _save(name, dict(mel=mel, moments=mom))


@torch.no_grad()
def gen_vocoder(R, name, cfg, B, frames):
    g = ref_vocoder(R, cfg["vocoder"])
    mel = cases.vocoder_input(cfg, B, frames)
    _save(name, dict(wave=g(mel)))


class _StubModel:
    """The attributes DDIMSampler touches (SURVEY.md 8c)."""

    def __init__(self, unet, tables):
        self.unet = unet
        self.num_timesteps = 1000
        self.parameterization = "eps"
        self.device = torch.device("cpu")
        for k, v in tables.items():
            setattr(self, k, v)

    def apply_model(self, x, t, c):
        return self.unet(x, t, y=c["y"], context_list=c["context_list"], context_attn_mask_list=c["mask_list"])

    def q_sample(self, x_start, t, noise=None):          # ddpm.py:430-436
        noise = torch.randn_like(x_start) if noise is None else noise
        a = self.sqrt_alphas_cumprod[t].reshape(-1, 1, 1, 1)
        b = self.sqrt_one_minus_alphas_cumprod[t].reshape(-1, 1, 1, 1)
        return a * x_start + b * noise


@torch.no_grad()
def gen_ddim(R, name, cfg, B, S, masked=False, with_audio=False, t5_len=32, audio_rows=None):
    m = ref_unet(R, cfg["unet"])
    tables = OF.ddpm_tables(cfg["linear_start"], cfg["linear_end"], cfg["timesteps"])
    stub = _StubModel(m, tables)
    sampler = R.DDIMSampler(stub, device=torch.device("cpu"))
    _, _, cond, unc = cases.unet_inputs(cfg, B, t5_len=t5_len)
    C, T, Fq = cfg["latent"]
    mask = x0 = None
    if masked:
        mask, x0 = cases.inpaint_mask(cfg, B)
    torch.manual_seed(cases.SAMPLER_SEED)
    t0 = time.time()
    sampler.make_schedule(ddim_num_steps=S, ddim_eta=1.0, verbose=False)
    img, _ = sampler.ddim_sampling(cond, (B, C, T, Fq), unconditional_guidance_scale=3.5,
                                   unconditional_conditioning=unc, mask=mask, x0=x0)
    print(f"  {name}: {S} steps in {time.time() - t0:.1f}s")
    out = dict(latent=img)
    if with_audio:
        dec, _, sd = ref_vae(R, cfg["vae"])
        h = torch.nn.functional.conv2d(img, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
        mel = dec(h)
        g = ref_vocoder(R, cfg["vocoder"])
        wave = g(mel.squeeze(1).permute(0, 2, 1))                 # ddpm.py:932-935
        if audio_rows is not None:       # large batches: keep the fixture small, store mel / waveform of a few rows only
            out["audio_rows"] = torch.tensor(audio_rows)
            mel, wave = mel[audio_rows], wave[audio_rows]
        out["mel"] = mel
        out["wave"] = wave
    _save(name, out)


@torch.no_grad()
def gen_stft(R, name, n_fft, hop, n_mels, sr, fmin, fmax, n_samples):
    st = R.TacotronSTFT(n_fft, hop, n_fft, n_mels, sr, fmin, fmax)
    wav = cases.wav_input(n_samples)
    mel, mag, _, _ = st.mel_spectrogram(wav)
    _save(name, dict(logmel=mel, mag_l2=torch.linalg.norm(mag)))


def gen_signatures(name):
    """Argument names and the source text of the defaults of the public pipeline functions (pipeline.py)."""
    src = open(os.path.join(ref_loader.REF_ROOT, "audioldm2", "pipeline.py")).read()
    out = {n.name: dict(args=[a.arg for a in n.args.args], defaults=[ast.get_source_segment(src, d) for d in n.args.defaults])
           for n in ast.parse(src).body
           if isinstance(n, ast.FunctionDef) and n.name in ("build_model", "text_to_audio", "super_resolution_and_inpainting")}
    path = os.path.join(HERE, name + ".json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {path}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    ap.add_argument("--skip-200", action="store_true")
    a = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    R = ref_loader.load()
    full, tiny, tinyf = arch.model_config("audioldm2-full"), arch.tiny_config(), arch.tiny_config(film=True)
    tinyl, tiny48 = arch.tiny_config(variant="large"), arch.tiny_config(variant="48k")
    m48, large = arch.model_config("audioldm_48k"), arch.model_config("audioldm2-full-large-1150k")
    jobs = {
        "unet_tiny_large": lambda: gen_unet(R, "unet_tiny_large", tinyl, 2, t5_len=5),
        "unet_tiny_48k": lambda: gen_unet(R, "unet_tiny_48k", tiny48, 2),
        "vae_tiny_48k": lambda: gen_vae(R, "vae_tiny_48k", tiny48, 2),
        "vocoder_tiny_48k": lambda: gen_vocoder(R, "vocoder_tiny_48k", tiny48, 2, 16),
        "unet_tiny": lambda: gen_unet(R, "unet_tiny", tiny, 2, t5_len=5),
        "unet_tiny_film": lambda: gen_unet(R, "unet_tiny_film", tinyf, 2),
        "vae_tiny": lambda: gen_vae(R, "vae_tiny", tiny, 2),
        "vocoder_tiny": lambda: gen_vocoder(R, "vocoder_tiny", tiny, 2, 24),
        "ddim_tiny": lambda: gen_ddim(R, "ddim_tiny", tiny, 2, 5, t5_len=5),
        "ddim_tiny_masked": lambda: gen_ddim(R, "ddim_tiny_masked", tiny, 2, 5, masked=True, t5_len=5),
        "stft_16k": lambda: gen_stft(R, "stft_16k", 1024, 160, 64, 16000, 0, 8000, 163840),
        "stft_tiny": lambda: gen_stft(R, "stft_tiny", 256, 40, 16, 4000, 0, 2000, 4000),
        "unet_full": lambda: gen_unet(R, "unet_full", full, 1),
        "vae_full": lambda: gen_vae(R, "vae_full", full, 1),
        "vocoder_full": lambda: gen_vocoder(R, "vocoder_full", full, 1, 1024),
        "ddim_full_10": lambda: gen_ddim(R, "ddim_full_10", full, 1, 10, with_audio=True),
        "ddim_full_200": lambda: gen_ddim(R, "ddim_full_200", full, 1, 200, with_audio=True),
        # round 2: the benchmark shape (B = 8), the other BASELINE configs at full size, a full-size masked run
        "unet_full_b8": lambda: gen_unet(R, "unet_full_b8", full, 8),
        "ddim_full_10_b8": lambda: gen_ddim(R, "ddim_full_10_b8", full, 8, 10, with_audio=True, audio_rows=[0, 7]),
        "ddim_full_200_b8": lambda: gen_ddim(R, "ddim_full_200_b8", full, 8, 200, with_audio=True, audio_rows=[0, 7]),
        "ddim_full_10_masked": lambda: gen_ddim(R, "ddim_full_10_masked", full, 1, 10, masked=True, with_audio=True),
        "unet_48k_full": lambda: gen_unet(R, "unet_48k_full", m48, 1),
        "vae_48k_full": lambda: gen_vae(R, "vae_48k_full", m48, 1),
        "vocoder_48k_full": lambda: gen_vocoder(R, "vocoder_48k_full", m48, 1, 1024),
        "unet_large_full": lambda: gen_unet(R, "unet_large_full", large, 1),
        "stft_48k": lambda: gen_stft(R, "stft_48k", 2048, 480, 256, 48000, 20, 24000, 491520),
        "pipeline_signatures": lambda: gen_signatures("pipeline_signatures"),
    }
    for k, fn in jobs.items():
        if a.only and k != a.only:
            continue
        if a.skip_200 and k in ("ddim_full_200", "ddim_full_200_b8"):
            continue
        print(k)
        fn()


if __name__ == "__main__":
    main()
