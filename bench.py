#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native AICoverGen hot path.

Metric (BASELINE.json): audio-seconds/sec (RTF) of the full cover pipeline on a 4-minute 44.1 kHz stereo song.
One "step" = one 4-min song through the song_cover_pipeline stage graph on one GPU:
    3 MDX-Net passes with denoise (Voc_FT / KARA_2 / Reverb_HQ-class geometries, 88+88+44x2 chunk inferences)
    -> mono 16 kHz -> VC.pipeline (HuBERT + rmvpe F0 + IVF index blend + flow/NSF-HiFiGAN synthesizer, 4 segments)
    -> vocal effects (high-pass, compressor, reverb) -> pydub mix (gains, overlay) -> the cover's int16 frames.
Weights are seeded synthetic checkpoints of the real architectures (no model files exist offline).
N GPUs = N songs (one per rank, weak scaling, no data-path collective).

  python bench.py --gpus 1 --steps 3 --warmup 3              # our arm
  python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR   # + the cover of the last timed step as DIR/*.npy
  python bench.py --impl reference --steps 1 --warmup 0      # CPU arm: the oracle restatement of the reference
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SONG_SECONDS = 240
SR = 44100
METRIC = "audio_seconds_per_second_full_cover_pipeline_4min_44k1_stereo"
DTYPE_NOTE = ("fp16 operands (MDX-Net U-Net, tcgen05 kind::f16) + tf32 (other tensor-core GEMMs; rmvpe as 3xTF32 split operands), fp32 "
              "accumulate; fp32/fp64 row kernels")
UNIT = "audio-s/s"
DUMP_FRAMES = 1 << 21               # --dump-outputs: at most this many cover frames (16 MB float32 + 16 MB of row numbers)


def synth_song(seconds: float, seed: int) -> np.ndarray:
    """SURVEY.md §8(d) cfg-4/5 style song: pink-ish noise bed + chord tones with slow AM + a vocal-like harmonic
    line with vibrato and unvoiced bursts, two decorrelated channels, peak 0.9."""
    rng = np.random.default_rng(seed)
    n = int(seconds * SR)
    t = np.arange(n, dtype=np.float64) / SR
    out = np.zeros((2, n))
    f0 = 220.0 * 2 ** (0.5 * np.sin(2 * np.pi * 0.2 * t)) * 2 ** (30 / 1200 * np.sin(2 * np.pi * 5.5 * t))
    ph = 2 * np.pi * np.cumsum(f0) / SR
    vocal = sum(np.sin(k * ph) / k for k in range(1, 9))
    burst = (t % 3.0) > 2.6
    vocal = np.where(burst, rng.standard_normal(n) * 0.5, vocal)
    vocal *= np.where((t % 7.3) > 6.9, 0.02, 1.0)
    for ch in range(2):
        white = rng.standard_normal(n)
        spec = np.fft.rfft(white)
        spec /= np.sqrt(np.maximum(np.arange(len(spec)), 1.0))
        bed = np.fft.irfft(spec, n)
        bed *= 0.25 / np.abs(bed).max()
        chord = sum(np.sin(2 * np.pi * f * (1 + 0.002 * ch) * t + ch) for f in (130.8, 164.8, 196.0))
        chord *= 0.15 * (0.6 + 0.4 * np.sin(2 * np.pi * 0.25 * t + ch))
        out[ch] = bed + chord + 0.35 * vocal * (1.0 - 0.1 * ch)
    out *= 0.9 / np.abs(out).max()
    return out.astype(np.float32)


# --------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                   capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.samples.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)

    def summary(self):
        sm = [float(s[1]) for s in self.samples if len(s) > 2 and s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if len(s) > 2 and s[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for nm, v in zip(names, s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------------------
def build_engine(device: str, rank_seed: int = 0):
    from aicovergen_b200.index import write_index_npz
    from aicovergen_b200.main import MDX_STAGES, CoverEngine
    from aicovergen_b200.synthetic import make_ivf_index_data

    hsd, rsd, cpt, mdx_w = bench_checkpoints()
    eng = CoverEngine(mdx_w, hsd, rsd, cpt, index=None, device=device)
    eng._rmvpe_sd = rsd
    # IVF index (README's IVF2237 example: 87 243 x 768) from HuBERT features of a seeded clip
    clip = torch.from_numpy(synth_song(20.0, 99).mean(0)[::3].copy())[None].to(device)     # crude 14.7 kHz stand-in clip
    feats = eng.hubert.extract_features(source=clip, padding_mask=None, output_layer=12)[0][0].cpu()
    cent, vecs = make_ivf_index_data(feats, n_total=87243, nlist=2237, lloyd=False)
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"b200vc_bench_index_{os.getpid()}.npz")
    write_index_npz(path, cent, vecs)
    eng.index_path = path
    return eng


def bench_checkpoints():
    """Seeded synthetic checkpoints of the real architectures, "trained-like": every BatchNorm carries the statistics of its
    own input on a seeded calibration clip (what training leaves behind) and the rmvpe head emits one smooth salience peak
    per frame, so activations, stems and F0 tracks have sane ranges (the raw random BatchNorm statistics of round 1 drove
    MDX activations to 1e5..1e10).  B200VC_RAW_CHECKPOINTS=1 restores the round-1 weights."""
    from aicovergen_b200.main import MDX_STAGES
    from aicovergen_b200.synthetic import (make_hubert_state_dict, make_mdx_state_dict, make_mdx_trained_like,
                                           make_rmvpe_state_dict, make_rmvpe_trained_like, make_rvc_checkpoint)

    raw = os.environ.get("B200VC_RAW_CHECKPOINTS") == "1"
    if raw:
        mdx_w = [make_mdx_state_dict(dim_f=s["dim_f"], dim_t=s["dim_t"], seed=2024 + i) for i, s in enumerate(MDX_STAGES)]
        rsd = make_rmvpe_state_dict()
    else:
        mdx_w = [make_mdx_trained_like(s["dim_f"], s["dim_t"], s["n_fft"], seed=2024 + i) for i, s in enumerate(MDX_STAGES)]
        rsd = make_rmvpe_trained_like()
    return make_hubert_state_dict(), rsd, make_rvc_checkpoint("40k", "v2"), mdx_w


def output_check(eng, song_dev, song_seconds):
    """Finite / non-silent check of every stem and of the cover produced by the graph that is being timed, plus the F0
    parity of the benchmarked utterance: coarse-pitch indices of the device rmvpe vs the CPU oracle on the SAME 16 kHz
    vocal the device pipeline converted (all frames of the padded utterance: 24 601 for a 4-min song)."""
    import scipy.signal as signal

    from aicovergen_b200 import ops
    from oracle import pipeline as opipe
    from oracle import rmvpe as orm

    def stat(t):
        t = t.float()
        return {"rms": round(float(t.pow(2).mean().sqrt()), 5), "peak": round(float(t.abs().max()), 4), "finite": bool(torch.isfinite(t).all())}

    stems = eng.separate(song_dev)
    res = {k: stat(v) for k, v in stems.items()}
    d = stems["dereverb"]
    mono = torch.empty(int(d.shape[1] * 16000 // 44100), device=d.device)
    ops.resample_sinc_mono(d.contiguous(), mono, 44100, 16000)
    ai = eng.convert(d, return_device=True)
    res["converted"] = stat(ai.float() / 32768.0)
    fx16 = eng.effects(ai)
    res["effected"] = stat(fx16.float() / 32768.0)
    cover = eng.mix(fx16, stems["backup"], stems["instrumental"])
    res["cover"] = stat(cover.float() / 32768.0)
    res["cover"]["frames"], res["cover"]["rate"] = int(cover.shape[0]), int(eng.cover_rate)
    bad = [k for k, v in res.items() if not v["finite"] or v["rms"] < 1e-4]
    if bad:
        raise SystemExit(f"bench: non-finite or silent output in {bad}: {res}")
    mono_h = mono.cpu().numpy()
    pad = np.pad(signal.filtfilt(opipe.bh, opipe.ah, mono_h), (48000, 48000), mode="reflect")
    pitch, pitchf = eng.vc.get_f0("bench", pad, len(pad) // 160, 0, "rmvpe", 3, 128)
    t0 = time.perf_counter()
    p_ref, pf_ref = orm.coarse_pitch(orm.infer_from_audio(eng._rmvpe_sd, pad.astype(np.float32), 0.03), 0)
    n = min(len(pitch), len(p_ref))
    res["f0_parity"] = {"frames": int(n), "coarse_pitch_mismatches": int((pitch[:n] != p_ref[:n]).sum()),
                        "voiced_frac": round(float((pf_ref[:n] > 0).mean()), 3), "distinct_levels": int(len(np.unique(p_ref[:n]))),
                        "oracle_cpu_s": round(time.perf_counter() - t0, 1)}
    return res


def dump_outputs(path, cover):
    """The cover's int16 frames [n, 2] as float32 `path`/cover.npy and their row numbers as float64 `path`/cover_frames.npy:
    all rows, or above DUMP_FRAMES a fixed seeded sample of them, so that two builds can be compared frame for frame."""
    os.makedirs(path, exist_ok=True)
    n = cover.shape[0]
    rows = np.arange(n) if n <= DUMP_FRAMES else np.sort(np.random.default_rng(0).choice(n, DUMP_FRAMES, replace=False))
    np.save(os.path.join(path, "cover.npy"), cover[rows].astype(np.float32))
    np.save(os.path.join(path, "cover_frames.npy"), rows.astype(np.float64))


def install_tc_profiler():
    """Wrap TapGemm.__call__ so every tcgen05 launch inside the timed region is bracketed by CUDA events on the
    launching stream; returns the record list [(kernel family, flops, bytes, start, end)]."""
    from aicovergen_b200 import tapgemm as tg

    records = []
    orig = tg.TapGemm.__call__

    def timed(self, stream=None, backend=None):
        be = self.backend if backend is None else backend
        if be == tg.BACKEND_TC and self.tc_supported() and install_tc_profiler.enabled:
            p = self.params
            if not hasattr(self, "_family"):
                tile_n = 256 if p.N > 128 else (128 if p.N > 64 else (64 if p.N > 32 else 32))
                # one family = one kernel template instance: tile width x operand type (kind::f16 and kind::tf32 are different
                # kernels with different rooflines)
                self._family = ("ws" if self.ws_applicable() else f"tc2<{tile_n}>") + ("/f16" if p.dtype & 1 else "/tf32")
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            orig(self, stream, backend)
            e.record()
            rows = p.OW * p.OH * p.OB
            es_in = self.a.t.element_size()
            es_out = self.out.t.element_size()
            flops = self.flops()
            if self.name in ("mdx.stft", "mdx.istft"):
                # a DFT restricted to dim_f bins run as a dense GEMM: count what an FFT of that frame would cost
                # (2.5 n log2 n real-FFT flops), not the 2*M*N*K of the GEMM, so the DFT does not inflate the roofline
                n_fft = p.Kc if self.name == "mdx.stft" else p.N
                flops = rows * 2.5 * n_fft * math.log2(n_fft)
            records.append((self._family, flops, float(rows) * (es_out * p.N + es_in * p.Kc), s, e, bool(p.dtype & 1), self.name))
        else:
            orig(self, stream, backend)

    tg.TapGemm.__call__ = timed
    install_tc_profiler.enabled = False
    return records


def host_cores() -> int:
    """CPU cores this process may actually use: affinity mask and cgroup quota, not the machine's core count
    (a 128-thread pool on a quota of a few cores makes the CPU arm pathologically slow)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
            quota = int(f.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
            period = int(f.read())
        if quota > 0:
            n = min(n, max(1, quota // period))
    except Exception:
        pass
    return max(1, n)


def best_cpu_threads() -> int:
    """The reference's CPU path gets the thread count that is actually fastest on this host (a short probe with a
    mid-size conv net): shared hosts often expose far more logical CPUs than a tenant can use productively."""
    from aicovergen_b200.synthetic import make_mdx_state_dict
    from oracle import mdx as om

    cores = host_cores()
    sd = make_mdx_state_dict(dim_f=512, dim_t=64, g=16, n=3)
    x = torch.randn(1, 4, 512, 64)
    best, best_t = cores, None
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores})
    for c in cands:
        torch.set_num_threads(c)
        om.convtdfnet(sd, x)
        t0 = time.perf_counter()
        om.convtdfnet(sd, x)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return d, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# --------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(threads: int, parts=None):
    """Times the CPU oracle (restatement of the reference, pinned against it) on a bounded sample and EXTRAPOLATES it to
    one 4-min song: per model one full-size chunk through STFT -> net -> iSTFT (x chunk count of a 4-min song with
    denoise), plus VC.pipeline with the 87 243-vector IVF index on 20 s (x 12).  Same checkpoints as the GPU arm.
    `parts`: which of the four parts (0-2: the MDX models, 3: VC.pipeline) to time NOW; the others reuse their latest timing
    (the reference arm rotates through the parts when it is asked for many steps, so that a 25-step run stays within minutes)."""
    from aicovergen_b200.main import MDX_STAGES
    from aicovergen_b200.synthetic import make_ivf_index_data
    from oracle import hubert as ohub
    from oracle import mdx as om
    from oracle import pipeline as opipe
    from oracle.index import IvfFlatIndex

    torch.set_num_threads(threads)
    hsd, rsd, cpt, mdx_w = bench_checkpoints()
    n_song = SONG_SECONDS * SR
    last = _CPU_CACHE.setdefault("part_s", {})
    todo = [p for p in range(4) if parts is None or p in parts or p not in last]
    measured = 0.0                     # CPU seconds actually spent in the timed parts of this sample
    detail = {}
    song = _CPU_CACHE.setdefault("song", synth_song(14.0, 1))
    chunks_of = {}
    for i, st in enumerate(MDX_STAGES):
        mp = om.MdxParams(st["dim_f"], st["dim_t"], st["n_fft"])
        gen = mp.chunk_size - mp.n_fft
        half = n_song // 2 + 44100
        chunks_of[i] = 2 * ((half + (gen - half % gen)) // gen)          # MDX.pad_wave per half (mdx.py:156-165)
        if i in todo:
            x = torch.from_numpy(song[:, :mp.chunk_size].copy())[None]
            t0 = time.perf_counter()
            om.convtdfnet(mdx_w[i], mp.stft(x))           # one chunk: STFT -> net
            mp.istft(mp.stft(x))                          #            -> iSTFT
            last[i] = time.perf_counter() - t0
            measured += last[i]
        detail[st["name"]] = {"s_per_chunk": round(last[i], 3), "chunks_per_sweep": chunks_of[i], "timed_this_step": i in todo}
    vc_s = 20
    if 3 in todo:
        if "index" not in _CPU_CACHE:          # index construction is model loading, not part of the timed conversion
            clip = torch.from_numpy(synth_song(20.0, 99).mean(0)[::3].copy())[None]
            feats = ohub.extract_features(hsd, clip, 12)[0]
            cent, vecs = make_ivf_index_data(feats, n_total=87243, nlist=2237, lloyd=False)
            _CPU_CACHE["index"] = IvfFlatIndex(cent, vecs)
        audio = synth_song(float(vc_s) * 44100 / 48000 + 1.0, 1).mean(0)[::3][: vc_s * 16000].astype(np.float32).copy()
        from oracle import effects as oeff
        from oracle import mixdown as omix
        oeff.build()
        stem16 = np.rint(synth_song(float(vc_s), 5) * np.float32(32767.0)).astype(np.int16).T.copy()      # [n, 2] @44.1k
        t0 = time.perf_counter()
        ai16 = opipe.pipeline(hsd, cpt, rsd, audio, index=_CPU_CACHE["index"], seed=0)
        fx16, _ = oeff.add_audio_effects(ai16, cpt["config"][-1], 0.15, 0.2, 0.8, 0.7)                   # main.py:206-226
        omix.combine_audio(fx16, cpt["config"][-1], stem16, 44100, stem16, 44100)                          # main.py:229-233
        last[3] = time.perf_counter() - t0
        measured += last[3]
    detail["vc_pipeline"] = {f"s_per_{vc_s}s_audio": round(last[3], 3), "index": "IVF2237 x 87243, index_rate 0.5", "timed_this_step": 3 in todo}
    total = sum(last[i] * chunks_of[i] * 2 for i in range(3)) + last[3] * (SONG_SECONDS / float(vc_s))   # denoise = 2 sweeps (mdx.py:261-263)
    detail["measured_cpu_s"] = round(measured, 2)
    detail["extrapolated_cpu_s_per_4min_song"] = round(total, 1)
    return SONG_SECONDS / total, total, detail


_CPU_CACHE: dict = {}


def run_reference(args, rank):
    if rank != 0:
        return
    threads = best_cpu_threads()
    if rank != 0:
        return
    vals = []
    n_all = max(args.warmup, 0) + max(args.steps, 1)
    rotate = n_all > 6                 # many steps requested: each step times ONE of the four parts, in rotation (~6 s per step)
    k = 0
    for _ in range(max(args.warmup, 0)):
        cpu_reference_sample(threads, [k % 4] if rotate else None)
        k += 1
    for _ in range(max(args.steps, 1)):
        v, tot, detail = cpu_reference_sample(threads, [k % 4] if rotate else None)
        k += 1
        vals.append((v, tot, detail))
    v = float(np.mean([x[0] for x in vals]))
    tot = float(np.mean([x[1] for x in vals]))
    meas = float(np.mean([x[2]["measured_cpu_s"] for x in vals]))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        # one step of this arm = one BOUNDED SAMPLE of the workload (that is what ran for ms_per_step); `value` is the
        # throughput of the full 4-min workload extrapolated from it (ms_per_full_step_extrapolated)
        "warmup": args.warmup, "ms_per_step": meas * 1000.0, "ms_per_full_step_extrapolated": tot * 1000.0,
        "sample_audio_seconds_equivalent": round(v * meas, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "song_cover_pipeline stage graph, 4-min 44.1 kHz stereo song (3 MDX passes w/ denoise + VC.pipeline rmvpe + effects + pydub mix), "
                               "CPU time extrapolated from a bounded sample", "sample": vals[-1][2]},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "EXTRAPOLATED: 1 full-size chunk per MDX model (STFT+net+iSTFT) x chunk count x2 sweeps, + VC.pipeline "
                                   "(rmvpe, IVF2237 x 87243 index) + effects + mix on 20 s x12; oracle/ restatement pinned against /root/reference",
                         "extrapolated": True},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------
# BASELINE.json configs 1-4 as separate bench lines (--config rmvpe10 | hubert30 | vc60 | mdx4min)
# --------------------------------------------------------------------------------------------------------------
def run_config(args, device):
    """One JSON line for one of BASELINE.json's per-operator configs: device-resident value, end-to-end value through the
    reference-facing array API (host buffers in, host result out), and the CPU oracle on the same input (bounded sample)."""
    from aicovergen_b200 import _ffi
    hsd, rsd, cpt, mdx_w = bench_checkpoints()
    name = args.config
    sr16 = 16000
    flush = torch.empty(256 * 1024 * 1024 // 4, device=device)
    cpu = None
    if name == "rmvpe10":
        from aicovergen_b200.rmvpe import RMVPEB200
        from oracle import rmvpe as orm
        seconds = 10.0
        t = np.arange(int(sr16 * seconds)) / sr16
        x = (0.5 * np.sin(2 * np.pi * (100 * t + 45 * t * t))).astype(np.float32)
        net = RMVPEB200(rsd, device=device)
        xd = torch.from_numpy(x).to(device)
        dev_fn = lambda: net.infer_from_audio_device(xd, 0.03)
        e2e_fn = lambda: net.infer_from_audio(x, 0.03)
        h2d, d2h = x.nbytes, 8 * (1 + len(x) // 160)
        cpu_fn, cpu_units = (lambda: orm.infer_from_audio(rsd, x, 0.03)), seconds
        workload = "cfg 1: rmvpe F0 on a 10 s 100->1000 Hz sine sweep @16 kHz (RMVPE.infer_from_audio, thred 0.03)"
    elif name == "crepe60":
        import types

        from aicovergen_b200.crepe import CrepeB200
        from aicovergen_b200.synthetic import make_crepe_state_dict
        from aicovergen_b200.vc_infer_pipeline import VC
        from oracle import crepe as oc
        seconds = 60.0
        x = synth_song(seconds * 44100 / 48000 + 1.0, 7).mean(0)[::3][: int(sr16 * seconds)].astype(np.float32).copy()
        csd = make_crepe_state_dict()
        vc = VC(40000, types.SimpleNamespace(device=device, is_half=True, x_pad=3, x_query=10, x_center=60, x_max=65))
        vc.model_crepe = CrepeB200(csd, device)
        xd = torch.from_numpy(x).to(device)
        dev_fn = lambda: vc.model_crepe.viterbi_bins(vc.model_crepe.activations(xd / float(np.quantile(np.abs(x), 0.999)), 128), 50.0, 1100.0)
        e2e_fn = lambda: vc.get_f0_crepe_computation(x.astype(np.float64), 50, 1100, None, 128)
        h2d, d2h = x.nbytes, 4 * (1 + len(x) // 128)
        cpu_fn, cpu_units = (lambda: oc.get_f0_crepe_computation(csd, x[: 4 * sr16].astype(np.float64), 50, 1100, None, 128)), 4.0
        workload = "crepe F0 (f0_method mangio-crepe, hop 128, torchcrepe 'full' CNN + Viterbi) on a 60 s vocal @16 kHz: 7501 frames, 21 TFLOP (CPU: 4 s)"
    elif name == "hubert30":
        from aicovergen_b200.hubert import HubertB200
        from oracle import hubert as ohub
        seconds = 30.0
        g = torch.Generator().manual_seed(0)
        n = int(sr16 * seconds)
        tt = torch.arange(n) / sr16
        x = (0.1 * torch.randn(n, generator=g) + 0.5 * torch.sin(2 * np.pi * (100 * tt + 15 * tt * tt))).float()[None]
        net = HubertB200(hsd, device)
        xd = x.to(device)
        dev_fn = lambda: net.extract_features(source=xd, padding_mask=None, output_layer=12)
        xp = x.pin_memory()
        e2e_fn = lambda: net.extract_features(source=xp.to(device, non_blocking=True), padding_mask=None, output_layer=12)[0].cpu()
        h2d, d2h = x.numel() * 4, 1499 * 768 * 4
        cpu_fn, cpu_units = (lambda: ohub.extract_features(hsd, x, 12)), seconds
        workload = "cfg 2: HuBERT-base layer-12 features of 30 s @16 kHz (extract_features, T = 1499)"
    elif name == "vc60":
        from aicovergen_b200 import rvc
        from aicovergen_b200.faiss_io import write_ivfflat
        from aicovergen_b200.rmvpe import RMVPEB200
        from aicovergen_b200.synthetic import make_ivf_index_data
        from oracle import pipeline as opipe
        seconds = 60.0
        x = synth_song(seconds * 44100 / 48000 + 1.0, 7).mean(0)[::3][: int(sr16 * seconds)].astype(np.float32).copy()
        cfg = rvc.Config(device, True)
        hub = rvc.load_hubert(device, True, {"model": hsd})
        cpt2, version, net_g, tgt_sr, vc = rvc.get_vc(device, True, cfg, dict(cpt))
        vc.model_rmvpe = RMVPEB200(rsd, device=device)
        clip = torch.from_numpy(synth_song(20.0, 99).mean(0)[::3].copy())[None].to(device)
        feats = hub.extract_features(source=clip, padding_mask=None, output_layer=12)[0][0].cpu()
        cent, vecs = make_ivf_index_data(feats, n_total=87243, nlist=2237, lloyd=False)
        from aicovergen_b200.index import write_index_npz
        path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"b200vc_bench_cfg3_{os.getpid()}.npz")
        write_index_npz(path, cent, vecs)
        xd = torch.from_numpy(x).to(device)
        call = lambda a: vc.pipeline(hub, net_g, 0, a, "x.wav", [0, 0, 0], 0, "rmvpe", path, 0.5, 1, 3, tgt_sr, 0, 0.25, version, 0.33, 128)

        def dev_fn():
            vc.return_device = True
            try:
                return call(xd)
            finally:
                vc.return_device = False
        e2e_fn = lambda: call(x)
        h2d, d2h = x.nbytes, 2399200 * 2
        cpu_fn, cpu_units = (lambda: opipe.pipeline(hsd, cpt, rsd, x[: 20 * sr16].copy(), index=None, seed=0)), 20.0
        workload = "cfg 3: VC.pipeline on a 60 s vocal, rvc.Config (3,10,60,65), rmvpe, IVF2237 x 87243 index_rate 0.5, v2 40k (CPU: 20 s, no index)"
    elif name == "mdx4min":
        from aicovergen_b200.mdx import MDX, MDXModel, run_mdx_arrays, run_mdx_device
        from oracle import mdx as om
        seconds = 240.0
        wave = synth_song(seconds, 0)
        sess = MDX(mdx_w[0], MDXModel(device, 3072, 256, 7680, stem_name="Vocals", compensation=1.009), int(device.split(":")[-1]))
        wd = torch.from_numpy(wave).to(device)
        dev_fn = lambda: run_mdx_device(sess, wd, denoise=False, m_threads=2)
        e2e_fn = lambda: run_mdx_arrays(sess, wave, denoise=False, m_threads=2)
        h2d, d2h = wave.nbytes, 2 * wave.nbytes
        mp = om.MdxParams(3072, 256, 7680)
        xc = torch.from_numpy(wave[:, :mp.chunk_size].copy())[None]
        cpu_fn = lambda: (mp.istft(om.convtdfnet(mdx_w[0], mp.stft(xc))))
        cpu_units = seconds / 44.0            # one of the 44 chunk inferences of the sweep
        workload = "cfg 4: mdx.run_mdx arithmetic (Kim_Vocal_2 geometry 3072x256/7680, denoise=False) on a 4-min 44.1 kHz stereo song, 44 chunk inferences (CPU: 1 chunk x44)"
    else:
        raise SystemExit(f"unknown --config {name}")

    def timed(fn, steps):
        tot = 0.0
        for _ in range(steps):
            flush.fill_(1.0)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            tot += s.elapsed_time(e)
        return tot

    for _ in range(max(args.warmup, 3)):
        dev_fn()
    sampler = ClockSampler(int(device.split(":")[-1]))
    sampler.start()
    l0 = _ffi.launch_count()
    dev_ms = timed(dev_fn, args.steps)
    launches = _ffi.launch_count() - l0
    e2e_fn()
    e2e_ms = timed(e2e_fn, args.steps)
    sampler.stop()
    line = {"metric": f"audio_seconds_per_second_{name}", "value": seconds * args.steps / (dev_ms / 1e3), "unit": UNIT, "n_gpus": 1,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "tf32/fp16 tensor-core GEMMs + fp32 row kernels", "data": "synthetic",
            "config": {"workload": workload, "l2": "256 MB buffer written between steps"}, "clocks": sampler.summary(),
            "e2e": {"value": seconds * args.steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches)}
    if not args.no_cpu_baseline:
        thr = best_cpu_threads()
        torch.set_num_threads(thr)
        t0 = time.perf_counter()
        cpu_fn()
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": cpu_units / dt, "unit": UNIT, "cores": thr, "kind": "port", "sample": f"{cpu_units:.1f} audio-s of the workload in {dt:.1f} s (oracle/)"}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seconds", type=float, default=float(SONG_SECONDS), help="song length (default: the 4-min headline config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="cover", choices=["cover", "rmvpe10", "hubert30", "vc60", "mdx4min", "crepe60"],
                    help="cover (default): the headline 4-min song_cover_pipeline graph; the others: BASELINE.json configs 1-4 as their own lines")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, BASELINE cfg 5): one song per GPU; strong (cfg 4 style): ONE song shared by all GPUs — MDX chunk "
                         "ranges per rank + all-gather, RVC segments round-robin after a broadcast F0")
    ap.add_argument("--no-output-check", action="store_true", help="skip the finite / non-silent / F0-parity check of the timed graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the cover returned by the last timed step to DIR (see dump_outputs); inputs and weights are seeded")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "cover"):
        ap.error("--dump-outputs writes the cover of the headline workload (--impl b200 --config cover)")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    from aicovergen_b200 import _ffi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (b200 arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    torch.cuda.manual_seed(0)          # the synthesizer's noise draws: the same outputs from run to run
    device = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    if args.config != "cover":
        if rank == 0:
            run_config(args, device)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    warm = max(args.warmup, 3)
    records = install_tc_profiler()
    eng = build_engine(device, rank)
    song = synth_song(args.seconds, seed=rank)
    song_pinned = torch.from_numpy(song).pin_memory()
    song_dev = song_pinned.to(device)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=device)        # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(fn, steps):
        """K steps, L2 flushed between steps, CUDA events on the launching stream, max over ranks."""
        total_ms = 0.0
        for _ in range(steps):
            flush.fill_(1.0)
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            total_ms += s.elapsed_time(e)
        t = torch.tensor([total_ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up (plan building, allocator growth, clocks)
    for _ in range(warm):
        eng.cover_device(song_dev)
    barrier()
    # ---- the graph being timed produces finite, non-silent stems and an F0 track that matches the CPU oracle (rank 0)
    checks = output_check(eng, song_dev, args.seconds) if (rank == 0 and not args.no_output_check) else None
    barrier()

    # ---- timed: inputs resident in HBM
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = _ffi.launch_count()
    dev_ms = timed_loop(lambda: eng.cover_device(song_dev), args.steps)
    launches = _ffi.launch_count() - l0
    # ---- timed: end to end through the public array API with HOST buffers (H2D of the song + D2H of the cover inside)
    out_host = {}
    cover_pinned = torch.empty((song.shape[1] + SR, 2), dtype=torch.int16).pin_memory()      # the caller's result buffer

    def e2e_step():
        out_host["cover"] = eng.cover(song_pinned.numpy(), out=cover_pinned)

    e2e_ms = timed_loop(e2e_step, args.steps)
    sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_host["cover"])
    # ---- one more step OUTSIDE the timed regions with CUDA events around every tcgen05 tap-GEMM launch (the event
    # pairs perturb launch overlap, so they must not sit inside the step timing): per-kernel-family roofline data
    from aicovergen_b200 import plans
    install_tc_profiler.enabled = True
    plans.graphs_enabled(False)            # the event pairs need the eager launch path (graph replays bypass Python)
    prof_ms = timed_loop(lambda: eng.cover_device(song_dev), 1)
    plans.graphs_enabled(True)
    install_tc_profiler.enabled = False

    # ---- strong scaling of ONE song over the N GPUs of the node (every rank holds the same song; MDX chunk ranges per rank +
    # one NCCL all-gather of the stem per pass; RVC: F0 on rank 0 -> broadcast -> segments round-robin -> all-gather of the PCM)
    strong = None
    if world > 1:
        song0 = torch.from_numpy(synth_song(args.seconds, seed=0)).to(device)
        for _ in range(3):          # plans / graphs for the sharded shapes
            eng.cover_device(song0, group=dist.group.WORLD)
        barrier()
        strong_ms = timed_loop(lambda: eng.cover_device(song0, group=dist.group.WORLD), args.steps)
        strong = {"value": args.seconds * args.steps / (strong_ms / 1000.0), "unit": UNIT, "ms_per_step": strong_ms / args.steps,
                  "songs": 1, "gpus": world,
                  "how": "one song on all GPUs: MDX chunk ranges per rank + all-gather of the stem per pass (3 passes), RVC F0 on "
                         "rank 0 -> broadcast -> <= n_segments ranks convert segments -> all-gather; time = max over ranks"}

    audio_s = args.seconds * world
    value = audio_s * args.steps / (dev_ms / 1000.0)
    e2e_value = audio_s * args.steps / (e2e_ms / 1000.0)

    # ---- roofline of the dominant kernel family (tcgen05 tap-GEMM, by tile width) and of the whole step
    pk, pk_src = peaks()
    f16_peak = pk["bf16_tflops_sustained"]            # fp16/bf16 dense, measured (sustained figure: kernels timed inside a long step)
    tf32_peak = f16_peak / 2.0                         # TF32 runs at half the fp16 rate on tcgen05 (nominal ratio; not measured separately)
    fam, layer = {}, {}
    for tile_n, fl, by, s, e, is_f16, lname in records:
        ms_i = s.elapsed_time(e)
        d = fam.setdefault(tile_n, [0.0, 0.0, 0.0, 0, 0.0])
        d[0] += ms_i
        d[1] += fl
        d[2] += by
        d[3] += 1
        d[4] += fl / (f16_peak if is_f16 else tf32_peak)          # roofline time of this launch, TFLOP / (TFLOP/s) units
        key = "".join("#" if c.isdigit() else c for c in lname)
        ly = layer.setdefault(key, [0.0, 0.0, 0])
        ly[0] += ms_i
        ly[1] += fl
        ly[2] += 1
    roof, step_roof = None, None
    traffic = None
    try:    # per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum, one ncu --set full capture) of the
            # representative launch of the dominant family: profiles/r02_dominant_traffic.json
        with open(os.path.join(ROOT, "profiles", "r02_dominant_traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass
    if fam:
        top = max(fam.items(), key=lambda kv: kv[1][0])
        tn, (ms, fl, by, cnt, roof_t) = top
        tot_ms = sum(v[0] for v in fam.values())
        tot_fl = sum(v[1] for v in fam.values())
        tot_roof = sum(v[4] for v in fam.values())
        top_layers = sorted(layer.items(), key=lambda kv: -kv[1][0])[:6]
        common = {"launches": cnt, "avg_launch_ms": round(ms / cnt, 4),
                  "share_of_step": round(ms / prof_ms, 4),
                  "algorithmic_tflops": round(fl / (ms / 1000.0) / 1e12, 2),
                  "algorithmic_gbs": round(by / (ms / 1000.0) / 1e9, 1),
                  "families_ms_per_step": {str(k): round(v[0], 2) for k, v in sorted(fam.items())},
                  "top_layers_ms": {k: {"ms": round(v[0], 2), "tflops": round(v[1] / v[0] / 1e9, 1), "launches": v[2]} for k, v in top_layers},
                  "profiled_step_ms": round(prof_ms, 1),
                  "flops_note": "2*M*N*K per tap-GEMM launch; the MDX STFT/iSTFT DFT-GEMMs are counted at FFT cost (2.5 n log2 n per frame)"}
        if traffic and traffic.get("family") == tn:
            common["traffic_detail"] = traffic
        if tn.startswith("ws") and fl / max(by, 1.0) < 100.0:
            # small-channel convolutions whose arithmetic intensity is below the machine balance -> HBM roofline
            achieved = by / (ms / 1000.0) / 1e9
            roof = {"kernel": f"tapgemm_ws_kernel [{tn}] (weight-stationary + halo, tcgen05.mma)", "bound": "hbm",
                    "achieved": round(achieved, 1), "peak": round(pk["hbm_gbs"], 1), "unit": "GB/s",
                    "frac": round(achieved / pk["hbm_gbs"], 4), "traffic": (traffic or {}).get("dram_bytes_per_launch") if (traffic or {}).get("family") == tn else None,
                    "peak_source": f"{pk_src} hbm_gbs", **common}
        else:
            achieved = fl / (ms / 1000.0) / 1e12
            eff_peak = fl / roof_t if roof_t > 0 else tf32_peak        # FLOP-weighted mix of the fp16 and TF32 peaks (TFLOP/s)
            roof = {"kernel": (f"tapgemm_ws_kernel [{tn}] (weight-stationary + halo, tcgen05.mma)" if tn.startswith("ws") else
                               f"tapgemm_tc2_kernel [{tn}] (persistent tcgen05.mma, double-buffered TMEM)"), "bound": "tensor",
                    "achieved": round(achieved, 2), "peak": round(eff_peak, 1), "unit": "TFLOP/s",
                    "frac": round(achieved / eff_peak, 4),
                    "traffic": (traffic or {}).get("dram_bytes_per_launch") if (traffic or {}).get("family") == tn else None,
                    "peak_source": f"{pk_src} bf16_tflops_sustained for kind::f16 kernels, half of it for kind::tf32 kernels "
                                   "(nominal 2:1; a TF32 peak is not in MEASURED_PEAKS.json)", **common}
        step_roof = {"tensor_tflop_per_step": round(tot_fl / 1e12, 2), "gemm_ms_per_step": round(tot_ms, 1),
                     "step_tflops": round(tot_fl / (prof_ms / 1000.0) / 1e12, 1),
                     "frac_of_tensor_roofline_whole_step": round((tot_roof * 1e-12 * 1000.0) / prof_ms, 4),
                     "frac_of_tensor_roofline_inside_gemms": round((tot_roof * 1e-12 * 1000.0) / tot_ms, 4),
                     "ms_outside_tcgen05_gemms": round(prof_ms - tot_ms, 1)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE_NOTE, "data": "synthetic",
            "config": {"workload": f"song_cover_pipeline stage graph on one {args.seconds:.0f}-s 44.1 kHz stereo song per GPU: 3 MDX-Net passes "
                                   "(3072x256/7680, 2048x256/5120, 3072x512/6144; denoise=True) + VC.pipeline (HuBERT-base, rmvpe, "
                                   "IVF2237 x 87243 index_rate 0.5, v2 40k synthesizer) + vocal effects (high-pass, compressor, reverb) "
                                   "+ pydub mix -> int16 cover frames",
                       "songs": world, "l2": "256 MB buffer written between steps; per-step working set >> 126 MB L2",
                       "weights": "seeded synthetic checkpoints of the real architectures, trained-like (BatchNorm statistics fitted on a calibration clip; smooth single-peak rmvpe salience)"},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(song.nbytes) * world,
                    "d2h_bytes_per_step": int(out_host["cover"].nbytes) * world, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches),
            "roofline": roof,
            "step_roofline": step_roof,
            "output_check": checks,
            "strong_scaling": strong,
        }
        if args.scaling == "strong" and strong is not None:
            line.update({"value": strong["value"], "ms_per_step": strong["ms_per_step"], "scaling": "strong",
                         "weak_scaling": {"value": value, "unit": UNIT, "ms_per_step": dev_ms / args.steps}})
            line["config"]["songs"] = 1
        if world == 1 and not args.no_cpu_baseline:
            thr = best_cpu_threads()
            v, tot, detail = cpu_reference_sample(thr)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": thr, "host_logical_cpus": host_cores(), "kind": "port", "extrapolated": True,
                                    "sample": "EXTRAPOLATED: 1 full-size chunk per MDX model x chunk count x2 sweeps + VC.pipeline (rmvpe, IVF index) on 20 s x12 (oracle/, pinned vs reference)",
                                    "detail": detail}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    try:
        os.unlink(eng.index_path)
    except OSError:
        pass


if __name__ == "__main__":
    main()
