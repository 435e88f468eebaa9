"""Bulk WAV ingest benchmark: extract_files(paths) against extract_many(16 kHz waves) on the same songs, and the batched
ingest kernel alone.

    python tools/bench_files.py [--songs 64] [--steps 3] [--seconds 240] [--out FILE]

Workload: N seeded songs (synth.tones), written as 44.1 kHz stereo s16 WAV files into a private temporary directory that
is removed on exit.  Every song is 10 584 000 frames = 3 840 000 samples at 16 kHz (BASELINE config 4).  The files are
written and then read by the same command, so they are read from the page cache, not from disk.

A/B legs alternate over --steps steps each.  The kernel leg times etude_ingest_pcm on all songs' raw bytes already on the
device (CUDA events; 2.7 GB at 64 songs, larger than the L2) and reports ms per audio-hour, GB/s of the algorithmic bytes
(raw in + 4 B out) and FMA/s of the taps the kernel visits, against the larger of the HBM floor (bytes over bench.peaks()
HBM) and the FMA floor (visited FMAs over 148 SMs x 128 lanes x the SM clock).  Prints one JSON line; --out also writes
it to FILE.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR_FILE = 44100


def gpu_info(index=0):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": q[0], "power_limit_w": float(q[1]), "sm_clock_max_mhz": float(q[2])}
    except Exception as e:   # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_clock_max_mhz": None, "note": str(e)}


def write_songs(tmp, n_songs, seconds):
    from etude_b200 import synth
    from scipy.io import wavfile
    n = SR_FILE * seconds
    # synth.tones costs ~1 s per audio-minute: ten-second seeded segments, tiled and shifted per song, plus seeded noise
    bases = [synth.tones(10 * SR_FILE, 1000 + k) for k in range(4)]
    paths = []
    for s in range(n_songs):
        rng = np.random.default_rng(s)
        mono = np.roll(np.tile(bases[s % 4], -(-n // len(bases[0])))[:n], 1237 * s) + rng.normal(0, 1e-3, n)
        st = np.stack([mono, mono * 0.7], axis=1)
        x = np.clip(np.round(st * 32767), -32768, 32767).astype(np.int16)
        p = os.path.join(tmp, f"song{s:03d}.wav")
        wavfile.write(p, SR_FILE, x)
        paths.append(p)
    return paths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--songs", type=int, default=64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--seconds", type=int, default=240)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_files needs a CUDA device")
    import bench
    import gpu_diag as D
    from etude_b200 import audio
    info = gpu_info()
    ex, _ = D.make_extractor(max_windows=32)
    eng = ex.engine
    tmp = tempfile.mkdtemp(prefix="etude_bench_files_")
    try:
        paths = write_songs(tmp, args.songs, args.seconds)
        infos = [audio.read_wav_info(p) for p in paths]
        n16 = int(eng.lib.etude_resampled_length(infos[0].n_frames, SR_FILE, 16000))
        assert n16 == 3840000 or args.seconds != 240, n16
        audio_s = sum(i.n_frames for i in infos) / SR_FILE
        # the 16 kHz waves of extract_many: the same songs through the device ingest (outside the timed legs)
        offs, total = audio.raw_layout(infos)
        host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        for i, o in zip(infos, offs):
            audio.read_wav_data(i, hv[o : o + i.data_bytes])
        raw_dev = host.to("cuda")
        wave_dev, wave_off, n_samples = eng.ingest_pcm(raw_dev, infos, 16000)
        waves = [wave_dev[o : o + n].cpu().numpy() for o, n in zip(wave_off, n_samples)]
        pinned = torch.empty(sum(n_samples), dtype=torch.float32, pin_memory=True)
        del wave_dev

        def leg_files():
            torch.cuda.synchronize()
            t = time.perf_counter()
            r = ex.extract_files(paths, as_dicts=False)
            torch.cuda.synchronize()
            return time.perf_counter() - t, r

        def leg_many():
            torch.cuda.synchronize()
            t = time.perf_counter()
            r = ex.extract_many(waves, as_dicts=False, pinned=pinned)
            torch.cuda.synchronize()
            return time.perf_counter() - t, r

        _, ra = leg_files()   # warm-up of both legs (module loads, allocator, tables)
        _, rb = leg_many()
        same = all(np.array_equal(a, b) for a, b in zip(ra, rb))
        t_files, t_many = [], []
        for _ in range(args.steps):
            t_files.append(leg_files()[0])
            t_many.append(leg_many()[0])

        # the kernel alone on device-resident raw bytes: per-launch CUDA events (host enqueue gaps excluded)
        n_ker = 10
        eng.ingest_pcm(raw_dev, infos, 16000)
        eng.profile_reset(timing=True)
        for _ in range(n_ker):
            eng.ingest_pcm(raw_dev, infos, 16000)
        prof = eng.profile_read()["ingest"]
        eng.profile_reset(timing=False)
        ms = prof["ms"] / n_ker
        prof = {k: v / n_ker for k, v in prof.items()}
        by, fl = prof["bytes"], prof["flops"]
        peaks = bench.peaks()
        clock = (info.get("sm_clock_max_mhz") or 1900.0) * 1e6
        fma_peak = 148 * 128 * clock
        floor_hbm = by / (peaks["hbm_gbs"] * 1e9) * 1e3
        floor_fma = (fl / 2) / fma_peak * 1e3
        res = {
            "metric": "bulk WAV ingest: extract_files vs extract_many, and the ingest kernel",
            "songs": args.songs, "song_seconds": args.seconds, "file_format": "44.1 kHz stereo s16 WAV",
            "files_read_from": "page cache (written by this command just before)",
            "audio_seconds": audio_s,
            "extract_files_audio_s_per_s": [audio_s / t for t in t_files],
            "extract_many_audio_s_per_s": [audio_s / t for t in t_many],
            "extract_files_over_extract_many": float(np.median(t_many) / np.median(t_files)),
            "same_records": bool(same),
            "h2d_bytes_extract_files": int(total), "h2d_bytes_extract_many": int(4 * sum(n_samples)),
            "kernel": {
                "ms_per_call": ms, "ms_per_audio_hour": ms / audio_s * 3600, "alg_bytes": by, "gb_per_s": by / ms / 1e6,
                "fma_visited": fl / 2, "fma_per_s": fl / 2 / ms * 1e3,
                "floor_hbm_ms": floor_hbm, "floor_fma_ms": floor_fma,
                "binding_floor": "hbm" if floor_hbm >= floor_fma else "fma",
                "share_of_binding_floor": max(floor_hbm, floor_fma) / ms,
                "hbm_peak": peaks, "fma_peak_per_s": fma_peak,
                "launches_per_call": prof["launches"],
            },
            **info,
        }
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
