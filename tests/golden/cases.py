"""Seeded inputs shared by the fixture generator and the tests (inputs are regenerated from
seeds; only reference OUTPUTS are stored in the .pt fixtures)."""
from __future__ import annotations

import os

import torch

from audioldm2_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
SAMPLER_SEED = 42          # pipeline.py:185 default seed
MAX_BYTES = 950_000        # every fixture file stays below 1 MB
BLOCK = 1024               # elements per kept block of a thinned tensor


def load(name: str) -> dict:
    return torch.load(os.path.join(HERE, name + ".pt"), map_location="cpu", weights_only=True)


def _cols(blocks: torch.Tensor, n: int) -> torch.Tensor:
    cols = (blocks[:, None] * BLOCK + torch.arange(BLOCK)).reshape(-1)
    return cols[cols < n]


def thin(d: dict, seed: int = 0) -> dict:
    """A fixture that would exceed MAX_BYTES keeps, of every float tensor of 64 Ki elements or more, the same seeded
    random subset of BLOCK-element blocks in each row (leading dimension): stored as [rows, kept elements], with the
    block indices under ``<key>_blocks``.  Tests compare through ``pick``."""
    size = lambda ks: sum(d[k].numel() * d[k].element_size() for k in ks)
    tensors = [k for k, v in d.items() if torch.is_tensor(v)]
    big = [k for k in tensors if d[k].is_floating_point() and d[k].numel() >= 1 << 16]
    if size(tensors) <= MAX_BYTES or not big:
        return d
    frac = (MAX_BYTES - 4096 * len(d) - (size(tensors) - size(big))) / size(big)     # 4 KB of archive overhead per entry
    g = torch.Generator().manual_seed(seed)
    out = dict(d)
    for k in big:
        x = d[k].reshape(d[k].shape[0], -1)
        nb = -(-x.shape[1] // BLOCK)
        blocks = torch.randperm(nb, generator=g)[:int(nb * frac)].sort().values
        out[k] = x[:, _cols(blocks, x.shape[1])].contiguous()
        out[k + "_blocks"] = blocks
    return out


def pick(g: dict, key: str, x: torch.Tensor) -> torch.Tensor:
    """The elements of ``x`` that fixture ``g`` stores for ``key``: all of them, or those ``thin`` kept."""
    blocks = g.get(key + "_blocks")
    if blocks is None:
        return x
    x = x.reshape(x.shape[0], -1)
    return x[:, _cols(blocks, x.shape[1]).to(x.device)]


def latent(cfg: dict, B: int, seed: int = 3) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    C, T, F = cfg["latent"]
    return torch.randn(B, C, T, F, generator=g)


def unet_inputs(cfg: dict, B: int, t5_len: int = 32, t_value: int = 501):
    x = latent(cfg, B, seed=3)
    t = torch.full((B,), t_value, dtype=torch.long)
    cond, unc = synth.conditioning(cfg, B, seed=77, t5_len=t5_len)
    return x, t, cond, unc


def mel_input(cfg: dict, B: int, seed: int = 9) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    C, T, F = cfg["latent"]
    ds = 2 ** (len(cfg["vae"]["ch_mult"]) - 1)
    return torch.randn(B, 1, T * ds, F * ds, generator=g)


def vocoder_input(cfg: dict, B: int, frames: int, seed: int = 11) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, cfg["vocoder"]["num_mels"], frames, generator=g)


def wav_input(n: int, seed: int = 13) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(1, n, generator=g) - 0.5)


def inpaint_mask(cfg: dict, B: int, seed: int = 15):
    """generate_batch_masked mask (ddpm.py:1611-1617): ones, zero over time rows [0.4,0.6)."""
    C, T, F = cfg["latent"]
    mask = torch.ones(B, 1, T, F)
    mask[:, :, int(T * 0.4):int(T * 0.6), :] = 0
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn(B, C, T, F, generator=g)
    return mask, x0


def sampler_noise(cfg: dict, B: int, S: int, masked: bool = False, seed: int = SAMPLER_SEED):
    """Replays the reference's CPU RNG draw order (SURVEY.md 7 H3): x_T (ddim.py:191), then per
    step [randn_like(x0) in q_sample when masked (ddpm.py:431)] and randn(shape) (ddim.py:351)."""
    C, T, F = cfg["latent"]
    torch.manual_seed(seed)
    x_T = torch.randn(B, C, T, F)
    noises, qn = [], []
    for _ in range(S):
        if masked:
            qn.append(torch.randn(B, C, T, F))
        noises.append(torch.randn(B, C, T, F))
    return x_T, noises, qn
