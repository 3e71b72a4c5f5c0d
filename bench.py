#!/usr/bin/env python
"""Benchmark of the AudioLDM2 sampling hot path (BASELINE.json metric: 10 s clips/sec @ 200 DDIM steps).

    python bench.py --gpus N --steps K --warmup W            # native sm_100a engine (one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own code on the host cores

A "step" is one pass of the hot path over one batch: x_T -> 200 x (cond+uncond UNet, CFG, DDIM update)
-> VAE decode -> HiFi-GAN -> waveform, for `--batch` prompts (config C2: audioldm2-full, batch 8).  Other BASELINE
configs: `--model audioldm_48k` (C3), `--model audioldm2-full-large-1150k` (C4), `--model audioldm_48k --mode
sr_inpainting` (C5: STFT/mel front end + VAE encoder + masked sampling).
Weights are the seeded synthetic checkpoint, conditioning is synthetic at the UNet boundary (no network: hub
checkpoints / tokenizers are unreachable; SURVEY.md 8d).  Conditioning encoders and the CLAP re-ranker are outside
the timed region (out of scope for this path).

The native arm (N = 1) also times, in the same process and on the same GPU, the reference's own PyTorch-CUDA path
(`torch_cuda_baseline`: unmodified reference modules from baseline/_ref when present, else the oracle port; two
apply_model calls per step as ddim.py:293-296) and reports `vs_torch_cuda` -- the north star's >= 4x target.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNIT = "clips/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--model", default="audioldm2-full")
    ap.add_argument("--mode", default="text_to_audio", choices=["text_to_audio", "sr_inpainting"])
    ap.add_argument("--batch", type=int, default=8, help="prompts per GPU (latent batch, n_candidate_gen_per_text=1)")
    ap.add_argument("--ddim-steps", type=int, default=200)
    ap.add_argument("--t5-len", type=int, default=32, help="Flan-T5 context length of the synthetic conditioning (SURVEY 8d: 32)")
    ap.add_argument("--lanes", type=int, default=None, help="UNet lanes (default: model.default_lanes / ALDM_LANES)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-pass", action="store_true")
    ap.add_argument("--no-torch-cuda-baseline", action="store_true")
    ap.add_argument("--ref-full", action="store_true", help="torch-CUDA baseline: run all DDIM steps for every precision mode")
    ap.add_argument("--dump-ops", default=None, help="write the per-op timing table of one UNet evaluation to this CSV")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the waveforms [clips, 1, samples] of the last timed step to DIR/wave.npy (float32; the leading clips "
                         "that fit in 64 MB): the inputs depend only on the arguments, so two builds can be compared output for output")
    return ap.parse_args()


def metric_name(a) -> str:
    m = f"10s clips/sec @{a.ddim_steps} DDIM steps ({a.model}"
    return m + (", sr_inpainting)" if a.mode == "sr_inpainting" else ")")


def workload(a, cfg) -> str:
    sr = cfg["sampling_rate"] // 1000
    w = (f"{a.model}, batch {a.batch} prompts/GPU, {a.ddim_steps} DDIM steps, 10 s @{sr} kHz, cfg 3.5, eta 1.0, "
         f"n_candidate_gen_per_text=1")
    if len([c for c in cfg["unet"]["context_dim"] if c is not None]):
        w += f", T5 len {a.t5_len}"
    if a.mode == "sr_inpainting":
        w += ", sr_inpainting: STFT/mel front end + VAE encoder + masked DDIM, time mask (0.40, 0.60)"
    return w


# ------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own modules (baseline/_ref) or the oracle port on the host cores.  Clips are independent,
# so the host is filled with W worker processes x T intra-op threads, each sampling B = 1.
# ------------------------------------------------------------------------------------------------
def _cpu_worker(conn, model_name, t5_len, threads, seed, cpus):
    # one block of logical CPUs per worker: without it the OpenMP runtimes of all workers may bind to the SAME cores
    # (measured on the 128-thread GPU-box host: 8 workers x 16 threads ran 10x slower than one worker alone)
    try:
        os.sched_setaffinity(0, cpus)
    except Exception:
        pass
    torch.set_num_threads(threads)
    from oracle import ref_bench
    ref = ref_bench.ReferencePath(model_name, 1, "cpu", t5_len=t5_len)
    conn.send(("ready", ref.kind, ref.where))
    while True:
        msg = conn.recv()
        if msg is None:
            return
        S, n_steps, with_decode = msg
        torch.manual_seed(seed)
        t0 = time.perf_counter()
        z = ref.sample(S, n_steps)
        t1 = time.perf_counter()
        if with_decode:
            ref.decode(z)
        t2 = time.perf_counter()
        conn.send((t1 - t0, (t2 - t1) if with_decode else None))


class CpuPool:
    def __init__(self, model_name: str, t5_len: int):
        import torch.multiprocessing as mp
        try:
            allowed = sorted(os.sched_getaffinity(0))
        except Exception:
            allowed = list(range(os.cpu_count() or 1))
        n = len(allowed)
        self.threads = int(os.environ.get("ALDM_CPU_THREADS", min(16, n)))
        self.workers = int(os.environ.get("ALDM_CPU_WORKERS", max(1, n // self.threads)))
        ctx = mp.get_context("spawn")
        self.conns, self.procs = [], []
        for w in range(self.workers):
            a, b = ctx.Pipe()
            cpus = set(allowed[(w * self.threads) % n:(w * self.threads) % n + self.threads]) or set(allowed)
            p = ctx.Process(target=_cpu_worker, args=(b, model_name, t5_len, self.threads, 1000 + w, cpus), daemon=True)
            p.start()
            self.conns.append(a); self.procs.append(p)
        infos = [c.recv() for c in self.conns]
        self.kind, self.where = infos[0][1], infos[0][2]
        self.t_dec = None
        self.active = self.workers
        self.calibration = None

    def calibrate(self, S: int):
        """How many of the spawned workers to run at once.  The logical-CPU count of a container says nothing about its CPU
        quota (the GPU box reports 128 logical CPUs; 8 concurrent 16-thread workers each ran 10x slower than one alone), so
        the whole-host throughput of 1, 2, 4, ... concurrent workers is measured on one DDIM step and the best count kept."""
        trials, k = {}, 1
        while True:
            self.active = min(k, self.workers)
            ps = self.run(S, 1, False)
            trials[self.active] = sum(1.0 / p for p in ps)
            if self.active == self.workers:
                break
            k *= 2
        self.active = max(trials, key=trials.get)
        self.calibration = {str(a): round(v, 4) for a, v in trials.items()}      # DDIM steps / s of the whole host
        if self.t_dec is not None:
            self.t_dec = self.t_dec[:self.active]

    def run(self, S: int, n_steps: int, with_decode: bool):
        conns = self.conns[:self.active]
        for c in conns:
            c.send((S, n_steps, with_decode))
        res = [c.recv() for c in conns]
        if with_decode:
            self.t_dec = [r[1] for r in res]
        return [r[0] / n_steps for r in res]             # seconds per DDIM step, per worker

    def clips_per_s(self, S: int, per_step) -> float:
        return sum(1.0 / (S * ps + td) for ps, td in zip(per_step, self.t_dec))

    def cores(self) -> int:
        return self.active * self.threads

    def describe(self, S, n_steps, per_step) -> str:
        return (f"{self.active} concurrent worker process(es) x {self.threads} threads, pinned to disjoint CPU blocks (host reports "
                f"{os.cpu_count()} logical CPUs; concurrency calibrated on whole-host DDIM steps/s: {self.calibration}), each B=1: "
                f"{n_steps} real DDIM steps (2 UNet calls each; mean {sum(per_step) / len(per_step):.2f} s/step) + VAE decode + HiFi-GAN "
                f"(mean {sum(self.t_dec) / len(self.t_dec):.2f} s, timed once), fp32 torch CPU, extrapolated to {S} steps per clip")

    def close(self):
        for c in self.conns:
            try:
                c.send(None)
            except Exception:
                pass
        for p in self.procs:
            p.join(10)


def run_reference_arm(a):
    """`--impl reference`: the reference's CPU implementation of the path, all host cores, bounded samples."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from audioldm2_b200 import arch
    cfg = arch.model_config(a.model)
    S = a.ddim_steps
    n_t = min(10, S)
    pool = CpuPool(a.model, a.t5_len)
    try:
        pool.run(S, 1, False)                                      # page in weights / thread pools
        pool.calibrate(S)
        for _ in range(a.warmup):
            pool.run(S, min(2, S), pool.t_dec is None)            # first warm-up also times the decode
        if pool.t_dec is None:
            pool.run(S, min(2, S), True)
        vals, last = [], None
        for _ in range(a.steps):
            last = pool.run(S, n_t, False)
            vals.append(pool.clips_per_s(S, last))
        v = sum(vals) / len(vals)
        line = dict(metric=metric_name(a), value=v, unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup,
                    ms_per_step=1000.0 * pool.active / v, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                    data="synthetic", impl="reference",
                    config=dict(workload=workload(a, cfg),
                                note="CPU arm: clips are independent, so each bench step times a bounded sample of this workload on every "
                                     "worker (see cpu_baseline.sample) and reports whole-host clips/s; text_to_audio path"),
                    cpu_baseline=dict(value=v, unit=UNIT, cores=pool.cores(), kind=pool.kind, where=pool.where,
                                      sample=pool.describe(S, n_t, last)),
                    e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
    finally:
        pool.close()


# ------------------------------------------------------------------------------------------------
# the reference's PyTorch-CUDA path on the same GPU (north star: "timed in the same run"; target >= 4x)
# ------------------------------------------------------------------------------------------------
def torch_cuda_baseline(a, dev, native_wave, seed):
    from oracle import ref_bench
    B, S = a.batch, a.ddim_steps
    ref = ref_bench.ReferencePath(a.model, B, dev, t5_len=a.t5_len)
    out = dict(kind=ref.kind, where=ref.where, batch=B, calls_per_step=2, ddim_steps=S)
    n_short = S if a.ref_full else min(20, S)
    rel = lambda x, y: float(torch.linalg.norm(x.double() - y.double()) / torch.linalg.norm(y.double()))
    waves = {}
    clocks = ClockSampler(dev.index or 0)
    clocks.start()
    for mode, n in (("high", S), ("default", n_short), ("fp32", S if native_wave is not None else n_short)):
        ref_bench.set_precision(mode)
        ref_bench.time_cuda(ref, S, 2)                                   # warm-up (cuDNN autotune, allocator)
        z, w, ts, td = ref_bench.time_cuda(ref, S, n if n < S else None, seed=seed)
        total = ts * (S / n) + td
        out[mode] = dict(value=B / total, unit=UNIT, ms_per_ddim_step=1e3 * ts / n, decode_ms=1e3 * td, steps_run=n,
                         extrapolated=n < S)
        if n >= S:
            waves[mode] = w
    out["clocks"] = clocks.stop()
    out["note"] = ("high = torch.set_float32_matmul_precision('high') as bin/audioldm2:139 sets it (TF32 matmuls + cuDNN TF32 convs): the "
                   "reference as shipped; default = torch defaults (TF32 convs, fp32 matmuls); fp32 = no TF32")
    if "fp32" in waves and "high" in waves:
        out["ref_high_vs_ref_fp32_wave_rel_l2"] = rel(waves["high"], waves["fp32"])
    if native_wave is not None and "fp32" in waves:
        out["native_vs_ref_fp32_wave_rel_l2"] = rel(native_wave, waves["fp32"])
        out["parity_note"] = (f"same seed ({seed}), same torch.randn draw order on the same CUDA generator, batch {B}, {S} steps: relative L2 of "
                              "the native waveform against the reference's fp32 CUDA waveform")
    return out


def kernel_pass(eng, peaks: dict, dump=None):
    """Per-launch CUDA-event timing of ONE UNet evaluation of one lane (eager, same stream), aggregated for the
    dominant kernel = gemm_tc3_kernel: achieved = sum(algorithmic FLOPs) / sum(durations)."""
    from audioldm2_b200 import _lib
    prog = eng.unet
    pl = prog.plan
    a, b = pl.marks["step_begin"], pl.marks["step_end"]
    h = prog.handles["step"]
    st = torch.cuda.current_stream()
    n = b - a
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
    for rep in range(2):                              # first repetition warms the caches / code
        evs[0].record(st)
        for i in range(n):
            _lib.check(prog.L.aldm_program_run_range(h, i, i + 1, st.cuda_stream), "run_range")
            evs[i + 1].record(st)
        st.synchronize()
    fl, tm, per_kind = 0.0, 0.0, {}
    for i in range(n):
        o = pl.ops[a + i]
        ms = evs[i].elapsed_time(evs[i + 1])
        per_kind[o["kind"]] = per_kind.get(o["kind"], 0.0) + ms
        if o["kind"] == "gemm":
            M = o["B"] * o["OH"] * o["OW"]
            fl += 2.0 * M * o["N"] * o["K"]
            tm += ms
    total = sum(per_kind.values())
    if dump:
        with open(dump, "w") as f:
            f.write("idx,kind,tag,ms,M,N,K,taps,splitk,bn,tflops\n")
            for i in range(n):
                o = pl.ops[a + i]
                ms = evs[i].elapsed_time(evs[i + 1])
                if o["kind"] == "gemm":
                    M = o["B"] * o["OH"] * o["OW"]
                    f.write(f"{i},gemm,{o['tag']},{ms:.4f},{M},{o['N']},{o['K']},{o['ntaps']},{o['splitk']},{o['bn']},"
                            f"{2.0 * M * o['N'] * o['K'] / (ms * 1e-3) / 1e12:.1f}\n")
                elif o["kind"] == "attn":
                    f.write(f"{i},attn,{o['tag']},{ms:.4f},{o['B'] * o['Nq']},{o['Nk']},{o['heads']},0,0,0,"
                            f"{4.0 * o['B'] * o['heads'] * o['Nq'] * o['Nk'] * 32 / (ms * 1e-3) / 1e12:.1f}\n")
                else:
                    f.write(f"{i},{o['kind']},{o.get('tag', 0)},{ms:.4f},{o.get('rows', 0)},{o.get('c0', 0)},0,0,0,0,0\n")
    peak = peaks.get("bf16_tflops_sustained") or 1432.6
    ach = fl / (tm * 1e-3) / 1e12 if tm > 0 else 0.0
    return dict(bound="tensor", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak, traffic=None,
                kernel="gemm_tc3_kernel (persistent tcgen05 implicit GEMM)", gemm_flop_per_lane_eval=fl,
                peak_source=("MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback"),
                share_of_unet_step={k: round(v / total, 4) for k, v in per_kind.items()},
                unet_eval_ms_eager=round(total, 3), lane_rows=pl.meta.get("Bt"))


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, wave, rank):
    """Rank 0 writes the waveforms of the whole batch (as many leading clips as fit in DUMP_BYTES) as float32."""
    if rank != 0:
        return
    import numpy as np
    row = wave[0].numel() * 4
    w = wave[:max(1, DUMP_BYTES // row)].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "wave.npy"), w)


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference_arm(a)
    from audioldm2_b200 import arch, engine, frontend, model, parallel, synth
    rank, world, local = parallel.init_from_env()
    assert torch.cuda.is_available(), "bench.py (native) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = arch.model_config(a.model)
    B, S = a.batch, a.ddim_steps
    sr_mode = a.mode == "sr_inpainting"
    eng = model.build_synthetic(a.model, batch=B, device=dev, t5_len=a.t5_len, use_graph=not a.no_graph, lanes=a.lanes,
                                with_encoder=sr_mode, arena_bcast=parallel.make_arena_bcast(dev) if world > 1 else None)
    # SURVEY 8e: the N-GPU job is the single-process batch of world*B prompts cut into contiguous shards -- conditioning and
    # noise are generated for the global batch from the same seeds on every rank and sliced
    Bg = world * B
    lo, hi = rank * B, (rank + 1) * B
    cond_g, unc_g = synth.conditioning(cfg, Bg, seed=77, t5_len=a.t5_len)
    cond_h, unc_h = parallel.shard_rows(cond_g, lo, hi), parallel.shard_rows(unc_g, lo, hi)
    pin = lambda c: dict(context_list=[t.pin_memory() for t in c["context_list"]], mask_list=[t.pin_memory() for t in c["mask_list"]],
                         y=None if c["y"] is None else c["y"].pin_memory())
    cond_h, unc_h = pin(cond_h), pin(unc_h)
    todev = lambda c: dict(context_list=[t.to(dev, non_blocking=True) for t in c["context_list"]],
                           mask_list=[t.to(dev, non_blocking=True) for t in c["mask_list"]],
                           y=None if c["y"] is None else c["y"].to(dev, non_blocking=True))
    cond_d, unc_d = todev(cond_h), todev(unc_h)
    C_, T, F_ = cfg["latent"]
    L = arch.vocoder_out_len(cfg["vocoder"], eng.mel_hw[0])
    wave_host = torch.empty(B, 1, L, dtype=torch.float32).pin_memory()
    guidance = 2.5 if sr_mode else 3.5            # pipeline.py:222 / :189 defaults
    wav_h = wav_d = mel_basis = mask = None
    if sr_mode:                                    # SURVEY 8d: 10.24 s of seeded uniform noise in [-0.5, 0.5] at the model rate
        vc = cfg["vocoder"]
        g = torch.Generator().manual_seed(13)
        wav_h = (torch.rand(Bg, eng.mel_hw[0] * vc["hop_size"], generator=g) - 0.5)[lo:hi].contiguous().pin_memory()
        wav_d = wav_h.to(dev)
        mel_basis = frontend.mel_basis_for(cfg).to(dev)
        mask = torch.ones(B, 1, T, F_, device=dev)
        mask[:, :, int(T * 0.40):int(T * 0.6), :] = 0

    def generate(seed, cond, unc, wav=None):
        sn = parallel.ShardedNoise(Bg, lo, hi, (C_, T, F_), dev, seed=seed)
        x0 = None
        if sr_mode:
            fb = engine.stft_mel(wav, vc["n_fft"], vc["hop_size"], mel_basis, out_frames=eng.mel_hw[0])       # K9
            mom = eng.encode_first_stage_moments(fb[:, None])
            pn = torch.randn(Bg, C_, T, F_, generator=torch.Generator().manual_seed(seed))[lo:hi]              # distributions.py:38 (CPU)
            x0 = eng.get_first_stage_encoding(mom, pn)
        return eng.generate_waveform(cond, unc, ddim_steps=S, guidance=guidance, eta=1.0, x_T=sn.x_T(), noise_fn=sn,
                                     mask=mask, x0=x0)

    def timed(fn, K):
        parallel.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            fn(i)
        e1.record()
        torch.cuda.synchronize(); parallel.barrier()
        return parallel.max_over_ranks(e0.elapsed_time(e1) * 1e-3, dev)

    for i in range(a.warmup):
        generate(1000 + i, cond_d, unc_d, wav_d)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # (1) device-resident: conditioning (and input audio) already in HBM, waveform left in HBM
    last = {}

    def dev_step(i):
        last["wave"] = generate(42 + i, cond_d, unc_d, wav_d)           # the engine's waveform slot: rewritten by the next call
    t_dev = timed(dev_step, a.steps)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, parallel.all_gather_rows(last["wave"], Bg), rank)

    # (2) end to end through the public seams: host conditioning / audio -> ... -> waveform in pinned host memory
    def e2e_step(i):
        w = generate(42 + i, todev(cond_h), todev(unc_h), wav_h.to(dev, non_blocking=True) if sr_mode else None)
        wave_host.copy_(w, non_blocking=True)
    t_e2e = timed(e2e_step, a.steps)
    clk = clocks.stop() if rank == 0 else None

    # phase breakdown + the waveform used for the parity figure against the reference's CUDA path (outside the timed regions)
    PSEED = 4242
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    native_wave = None
    if not sr_mode:
        sn = parallel.ShardedNoise(Bg, lo, hi, (C_, T, F_), dev, seed=PSEED)
        ev[0].record(); z = eng.generate_latent(cond_d, unc_d, ddim_steps=S, guidance=guidance, eta=1.0, x_T=sn.x_T(), noise_fn=sn)
        ev[1].record(); mel = eng.decode_first_stage(z)
        ev[2].record(); native_wave = eng.mel_spectrogram_to_waveform(mel).clone()
        ev[3].record(); torch.cuda.synchronize()
        breakdown = dict(sampler_ms=ev[0].elapsed_time(ev[1]), vae_decode_ms=ev[1].elapsed_time(ev[2]),
                         vocoder_ms=ev[2].elapsed_time(ev[3]), ms_per_ddim_step=ev[0].elapsed_time(ev[1]) / S)
    else:
        ev[0].record(); fb = engine.stft_mel(wav_d, vc["n_fft"], vc["hop_size"], mel_basis, out_frames=eng.mel_hw[0])
        ev[1].record(); eng.encode_first_stage_moments(fb[:, None])
        ev[2].record(); generate(PSEED, cond_d, unc_d, wav_d)
        ev[3].record(); torch.cuda.synchronize()
        breakdown = dict(stft_mel_ms=ev[0].elapsed_time(ev[1]), vae_encode_ms=ev[1].elapsed_time(ev[2]),
                         whole_generate_ms=ev[2].elapsed_time(ev[3]))

    clips = world * B * a.steps
    lanes_used = eng.lanes
    value, e2e_value = clips / t_dev, clips / t_e2e
    h2d = sum(t.numel() * 4 for c in (cond_h, unc_h) for t in c["context_list"] + c["mask_list"]) + \
        sum(c["y"].numel() * 4 for c in (cond_h, unc_h) if c["y"] is not None) + (wav_h.numel() * 4 if sr_mode else 0)
    per_gen = S * eng.launches_per_step() + eng.launches_decode() + eng.launches_cond()
    if sr_mode:
        per_gen += 1 + eng.vae_enc.num_launches("all") + 1 + S          # K9, encoder, posterior, masked blend per step
    launches = a.steps * per_gen
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    roof = None if a.no_kernel_pass else kernel_pass(eng, peaks, a.dump_ops)
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if roof is not None:
            roof["traffic"] = tr.get("gemm_tc_kernel_dram_bytes_per_launch")
            roof["traffic_source"] = tr.get("source", "profiles/traffic.json")
    except Exception:
        pass
    if roof is not None and breakdown.get("ms_per_ddim_step"):
        # `achieved` divides by per-op event times of an EAGER pass of one lane (every op carries a launch gap).  The same FLOPs
        # (all lanes) over the whole measured graph-replay step -- GEMMs, attention, norms and gaps included -- bound it from below.
        g = float(breakdown["ms_per_ddim_step"])
        roof["gemm_tflops_over_whole_step"] = round(roof["gemm_flop_per_lane_eval"] * lanes_used / (g * 1e-3) / 1e12, 2)
    cpu = None
    if world == 1 and not a.no_cpu_baseline and not sr_mode:
        pool = CpuPool(a.model, a.t5_len)
        try:
            pool.run(S, 1, False)
            pool.calibrate(S)
            pool.run(S, 1, True)
            ps = pool.run(S, min(10, S), False)
            cpu = dict(value=pool.clips_per_s(S, ps), unit=UNIT, cores=pool.cores(), kind=pool.kind, where=pool.where,
                       sample=pool.describe(S, min(10, S), ps))
        finally:
            pool.close()
    tcb = None
    if world == 1 and not a.no_torch_cuda_baseline and not sr_mode:
        nw = native_wave
        del eng
        torch.cuda.empty_cache()
        try:
            tcb = torch_cuda_baseline(a, dev, nw, PSEED)
        except Exception as e:      # the baseline leg must never take the native line down
            tcb = dict(error=repr(e))
    line = dict(metric=metric_name(a), value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
                ms_per_step=1000.0 * t_dev / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f16x2 (split-fp16 tensor-core operands: weights hi + lo, activations hi + lo in the convolutions and one plane on the token side; fp32 accumulate, fp32 residual stream)", data="synthetic",
                config=dict(workload=workload(a, cfg), lanes=lanes_used,
                            l2="no explicit flush: the UNet weights (1.39 GB for audioldm2-full) are re-streamed every DDIM step "
                               "(working set >> 126 MB L2)",
                            parallelism=f"dp{world} (contiguous shards of the global batch of {Bg}, weights broadcast once over NCCL, "
                                        "no per-step collective)"),
                e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=wave_host.numel() * 4),
                gpu_launches=launches, clocks=clk, roofline=roof, cpu_baseline=cpu, impl="native", breakdown=breakdown)
    if tcb is not None:
        line["torch_cuda_baseline"] = tcb
        if "high" in tcb:
            line["vs_torch_cuda"] = dict(ratio=value / tcb["high"]["value"], e2e_ratio=e2e_value / tcb["high"]["value"],
                                         against="high (the reference as shipped: TF32 matmuls + TF32 convs)",
                                         ratio_vs_default=value / tcb["default"]["value"], ratio_vs_fp32=value / tcb["fp32"]["value"])
    print(json.dumps(line))


if __name__ == "__main__":
    try:
        main()
    finally:
        import torch.distributed as _dist
        if _dist.is_available() and _dist.is_initialized():
            _dist.destroy_process_group()
