"""CPU tests of the host-side mirror of the reference interface: pipeline signatures and defaults (pipeline.py:142-267),
DiffusionWrapper.forward's cond-dict unpacking (ddpm.py:1821-1879), the n_gen tiling / candidate selection of
generate_batch (ddpm.py:1516-1525,1554-1564), package exports (audioldm2/__init__.py:1-2), save_wave, the mel
filterbank against independent golden values, and the multi-rank noise sharding rule (SURVEY.md 8e)."""
import inspect
import os
import wave

import numpy as np
import pytest
import torch

import audioldm2_b200 as A
from audioldm2_b200 import frontend, model, parallel, pipeline
from tests.golden import cases

# pipeline.py:142, :181-193, :213-230 -- argument names in positional order and their defaults
REF_SIGNATURES = {
    "build_model": (["ckpt_path", "config", "device", "model_name"], [None, None, None, "audioldm2-full"]),
    "text_to_audio": (["latent_diffusion", "text", "transcription", "seed", "ddim_steps", "duration", "batchsize", "guidance_scale",
                       "n_candidate_gen_per_text", "latent_t_per_second", "config"],
                      ["", 42, 200, 10, 1, 3.5, 3, 25.6, None]),
    "super_resolution_and_inpainting": (["latent_diffusion", "text", "transcription", "original_audio_file_path", "seed", "ddim_steps",
                                         "duration", "batchsize", "guidance_scale", "n_candidate_gen_per_text",
                                         "time_mask_ratio_start_and_end", "freq_mask_ratio_start_and_end", "latent_t_per_second",
                                         "config"],
                                        ["", None, 42, 200, None, 1, 2.5, 3, (0.40, 0.6), (1.0, 1.0), 25.6, None]),
}


@pytest.mark.parametrize("name", sorted(REF_SIGNATURES))
def test_signatures_match_reference(name):
    names, defaults = REF_SIGNATURES[name]
    pos = [p for p in inspect.signature(getattr(A, name)).parameters.values() if p.kind == p.POSITIONAL_OR_KEYWORD]
    assert [p.name for p in pos] == names
    assert [p.default for p in pos if p.default is not p.empty] == defaults


def test_signatures_against_reference_source_when_present():
    """REF_SIGNATURES against the signatures parsed from the reference's pipeline.py (tests/golden/make_golden.py)."""
    import ast
    import json
    with open(os.path.join(cases.HERE, "pipeline_signatures.json")) as f:
        ref = json.load(f)
    assert sorted(ref) == sorted(REF_SIGNATURES)
    for name, sig in ref.items():
        assert sig["args"] == REF_SIGNATURES[name][0]
        assert [ast.literal_eval(d) for d in sig["defaults"]] == REF_SIGNATURES[name][1]


def test_package_exports():
    for n in ("seed_everything", "save_wave", "get_time", "get_duration", "read_list",          # audioldm2/__init__.py:1
              "build_model", "text_to_audio", "super_resolution_and_inpainting"):                 # pipeline.*
        assert callable(getattr(A, n))


def test_unpack_cond_dict_film_and_crossattn_order():
    B = 3
    y1, y2 = torch.randn(B, 1, 4), torch.randn(B, 1, 2)
    c1, m1 = torch.randn(B, 8, 6), torch.ones(B, 8)
    c2, m2 = torch.randn(B, 5, 7), torch.ones(B, 5)
    d = {"film_clap": y1, "crossattn_a": [c1, m1], "noncond_loss": torch.zeros(1), "film_b": y2, "crossattn_b": (c2, m2)}
    u = model.unpack_cond_dict(d)
    assert torch.equal(u["y"], torch.cat([y1.squeeze(1), y2.squeeze(1)], -1))                     # ddpm.py:1836-1840
    assert u["context_list"][0] is c1 and u["context_list"][1] is c2 and u["mask_list"][1] is m2
    # the conditioning_key order, not the dict order, decides (reorder_cond_dict, ddpm.py:1028-1032)
    r = model.unpack_cond_dict(model.reorder_cond_dict(d, ["crossattn_b", "crossattn_a", "film_clap"]))
    assert r["context_list"][0] is c2 and r["context_list"][1] is c1 and torch.equal(r["y"], y1.squeeze(1))
    # dict-valued entry: the LAST inner crossattn* pair wins (ddpm.py:1843-1848)
    inner = {"crossattn_x": [c1, m1], "other": 1, "crossattn_y": [c2, m2]}
    v = model.unpack_cond_dict({"crossattn_seq": inner})
    assert v["context_list"] == [c2] and v["mask_list"] == [m2] and v["y"] is None
    with pytest.raises(NotImplementedError):
        model.unpack_cond_dict({"bogus": c1})
    # already-unpacked dicts pass through
    w = model.unpack_cond_dict(dict(context_list=[c1], mask_list=[m1], y=None))
    assert w["context_list"][0] is c1


def test_tile_and_select_best_follow_generate_batch():
    B, n_gen = 2, 3
    c = dict(context_list=[torch.arange(B).float().reshape(B, 1, 1)], mask_list=[torch.ones(B, 1)], y=None)
    t = pipeline._tile(c, n_gen)
    assert t["context_list"][0].reshape(-1).tolist() == [0, 1, 0, 1, 0, 1]                        # rows i + k*B (ddpm.py:1516-1525)
    wav = np.arange(B * n_gen, dtype=np.float32).reshape(B * n_gen, 1, 1)
    sim = torch.tensor([0.1, 0.9, 0.5, 0.2, 0.3, 0.95])                                           # prompt 0: rows 0,2,4; prompt 1: rows 1,3,5
    out, idx = pipeline.select_best(wav, sim, B)
    assert idx == [2, 5] and out.reshape(-1).tolist() == [2.0, 5.0]                               # ddpm.py:1559-1564


def test_make_batch_and_save_wave(tmp_path):
    b = pipeline.make_batch_for_text_to_audio("a dog", batchsize=2)
    assert b["text"] == ["a dog", "a dog"] and b["fname"] == ["a_dog", "a_dog"] and tuple(b["log_mel_spec"].shape) == (2, 1024, 64)
    w = (np.sin(np.linspace(0, 20, 1600)) * 0.5).astype(np.float32)[None, None].repeat(2, 0)
    paths = A.save_wave(w, str(tmp_path), name="x")
    assert [os.path.basename(p) for p in paths] == ["x_0.wav", "x_1.wav"]                         # utils.py:58-63
    assert abs(A.get_duration(paths[0]) - 0.1) < 1e-6
    x, sr = frontend.read_wav(paths[1])
    assert sr == 16000 and np.abs(x - w[1, 0]).max() < 1.0 / 32767
    (p,) = A.save_wave(w[:1], str(tmp_path), name="single")
    assert os.path.basename(p) == "single.wav"
    with wave.open(p) as f:
        assert f.getsampwidth() == 2 and f.getnchannels() == 1


def test_mel_basis_matches_independent_golden():
    g = torch.load(os.path.join(cases.HERE, "mel_basis.pt"), weights_only=True)
    for name, d in g.items():
        sr, n_fft, n_mels, fmin, fmax = d["args"].tolist()
        mine = frontend.mel_basis(int(sr), int(n_fft), int(n_mels), fmin, fmax)
        gold = torch.zeros(tuple(d["shape"].tolist()))
        gold[d["nz_index"][0].long(), d["nz_index"][1].long()] = d["nz_value"]
        assert mine.shape == gold.shape
        assert float((mine - gold).abs().max()) < 1e-7 * float(gold.abs().max()) + 1e-9, name
        assert d["torchaudio_max_dev"] < 1e-6


def test_prepare_waveform_follows_read_wav_file():
    g = np.random.default_rng(0)
    x = g.normal(size=3000).astype(np.float32) + 0.3
    y = frontend.prepare_waveform(x, 16000, 16000, 4000)                                          # tools.py:28-40
    assert y.shape == (1, 4000) and abs(np.abs(y).max() - 0.5) < 1e-6 and np.all(y[0, 3000:] == 0)
    z = frontend.prepare_waveform(x, 16000, 16000, 2000)
    assert z.shape == (1, 2000) and abs(np.abs(z).max() - 0.5) < 1e-6


def test_sharded_noise_reproduces_single_process_batch():
    latent = (2, 4, 3)
    full = parallel.ShardedNoise(6, 0, 6, latent, "cpu", seed=42)
    parts = [parallel.ShardedNoise(6, lo, hi, latent, "cpu", seed=42) for lo, hi in ((0, 2), (2, 4), (4, 6))]
    for draw in ("x_T", "q", "step", "q", "step"):
        ref = full.x_T() if draw == "x_T" else full(0, draw)
        got = torch.cat([p.x_T() if draw == "x_T" else p(0, draw) for p in parts])
        assert torch.equal(got, ref)
    # ... and the unsharded object equals the reference's plain torch.randn sequence on the default generator
    torch.manual_seed(42)
    one = parallel.ShardedNoise(6, 0, 6, latent, "cpu", seed=42)
    assert torch.equal(one.x_T(), torch.randn(6, *latent)) and torch.equal(one(0, "step"), torch.randn(6, *latent))
    c = dict(context_list=[torch.arange(6).float().reshape(6, 1, 1)], mask_list=[torch.ones(6, 1)], y=None)
    s = parallel.shard_rows(c, 2, 4)
    assert s["context_list"][0].reshape(-1).tolist() == [2.0, 3.0] and s["y"] is None
