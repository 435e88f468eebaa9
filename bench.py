#!/usr/bin/env python
"""Extract-stage throughput benchmark (BASELINE.json: audio-seconds per second at 1/2/4/8 B200; % of tensor / HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 4|3|2] [--impl reference] [--dump-outputs DIR]

One *step* = the whole hot path over the workload: fused log-mel front-end -> every 512-frame window through the
hFT-Transformer -> piano-rolls stitched on the device -> device note decoding -> note records on the host.

  --config 4 (default)  BASELINE config 4: "extractor over 256 synthetic 4-min songs sharded by window across 1/2/4/8 B200":
                        the FIXED 256-song job, 256 / N songs per rank (strong scaling), window batch 32, no collective on
                        the hot path; the e2e leg runs `sharding.extract_sharded` and ends with the one final gather of the
                        note records to rank 0 (NCCL, device to device, then one copy to the host).
  --config 3            BASELINE config 3: "full extractor on one 4-min synthetic song, 1 B200, bf16, window batch 64"
                        (30 windows = one batch).  With --gpus N > 1 the song's windows are split over the ranks and the
                        rolls gathered (`sharding.extract_window_sharded`).
  --config 2            BASELINE config 2: the log-mel front-end alone over 10 h of synthetic audio (HBM roofline).  The
                        default run also carries this measurement in its `frontend_10h` object.

Printed JSON (rank 0): `value` = audio-s/s of the whole path with the waves already resident in HBM (log-mel + model +
note decoding, note records back on the host); `e2e` = the same through the public API with pinned HOST waves in (H2D
inside the timed region) and, for N > 1, the final gather; `roofline` = the dominant kernel class (CUDA-event timed inside
a separate profiled pass of the device leg) against the measured bf16 peak; `frontend` / `frontend_10h` = the log-mel
kernel against the measured HBM peak; `cpu_baseline` = the oracle port (torch CPU restatement of the reference) on this
box's host cores over a bounded sample.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned as DIR/<name>.npy (float64 or
float32, under 64 MB in all; see `dump_notes` / `dump_features`).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 16000
SONG_SECONDS = 240
SONG_SAMPLES = SR * SONG_SECONDS
TOTAL_SONGS = 256
FLOP_PER_WINDOW_REF = 1050.9e9       # reference formulation (SURVEY.md 8(a)); executed count comes from the library
METRIC = "extract_throughput_audio_seconds_per_second"
UNIT = "audio-s/s"
CONFIG_TEXT = {
    4: "extractor over 256 synthetic 4-min songs sharded by window across 1/2/4/8 B200",
    3: "full extractor on one 4-min synthetic song, 1 B200, bf16, window batch 64",
    2: "log-mel STFT front-end microbench over 10 h of synthetic audio on 1 B200 (HBM-bound)",
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_burst": p["bf16_tflops"], "bf16_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 4:] if sm else []   # drop idle samples before the first launch
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_wave(song_index, n_samples=SONG_SAMPLES):
    from etude_b200 import synth
    return synth.noise(n_samples, seed=1234 + song_index)


DUMP_RECORDS = 1 << 20      # note records kept by --dump-outputs: 6 float64 columns, 48 MB at most
DUMP_ROWS = 16384           # log-mel rows kept by --dump-outputs of config 2: 16 MB of float32


def dump_notes(out_dir, recs, song_ids):
    """--dump-outputs of configs 4 and 3: the note records (what extract_many(as_dicts=False) returns) of rank 0's songs.
    note_counts.npy: the record count of each song, in the order of `song_ids`; note_{song,index,pitch,velocity,onset,
    offset}.npy: every record when all songs together hold at most DUMP_RECORDS, else DUMP_RECORDS / len(recs) records per
    song at sorted positions drawn by a generator seeded with the song's index.  The positions depend only on the song and
    its record count, so two builds that compute the same notes write identical files."""
    os.makedirs(out_dir, exist_ok=True)
    counts = [len(r) for r in recs]
    per_song = sum(counts) if sum(counts) <= DUMP_RECORDS else DUMP_RECORDS // len(recs)
    cols = {k: [np.zeros(0)] for k in ("song", "index", "pitch", "velocity", "onset", "offset")}
    for s, r in zip(song_ids, recs):
        n = len(r)
        idx = np.arange(n) if n <= per_song else np.sort(np.random.default_rng(s).choice(n, per_song, replace=False))
        cols["song"].append(np.full(len(idx), s))
        cols["index"].append(idx)
        for k in ("pitch", "velocity", "onset", "offset"):
            cols[k].append(r[k][idx])
    np.save(os.path.join(out_dir, "note_counts.npy"), np.asarray(counts, np.float64))
    for k, v in cols.items():
        np.save(os.path.join(out_dir, f"note_{k}.npy"), np.concatenate(v).astype(np.float64))


def dump_features(out_dir, feat):
    """--dump-outputs of config 2: DUMP_ROWS rows of the last launch's log-mel features, at sorted positions drawn by a
    generator seeded with 0 (logmel_rows.npy, float64), and those rows (logmel.npy, float32 [DUMP_ROWS, 256])."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(feat.shape[0], min(DUMP_ROWS, feat.shape[0]), replace=False))
    np.save(os.path.join(out_dir, "logmel_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "logmel.npy"), feat[torch.from_numpy(rows).to(feat.device)].float().cpu().numpy())


def cpu_baseline_sample(threads, windows=4, repeats=1):
    """Oracle port (torch fp32 CPU restatement of the reference extractor) on a bounded sample: log-mel + `windows`
    windows + note decoding of one synthetic clip.  Returns (audio-s/s, description)."""
    from etude_b200 import synth
    from oracle import logmel as ologmel
    from oracle import model as omodel
    from oracle import notes as onotes
    torch.set_num_threads(threads)
    sd = omodel.init_state_dict(0)
    n = 256 * (512 * windows - 1)
    wave = synth.noise(n, 1234)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        feat = ologmel.logmel(wave, dtype=np.float32)
        outs = omodel.transcript(sd, feat, batch=windows)
        onotes.mpe2note(outs[4], outs[5], outs[6], outs[7], 0.5, 1.0, 0.5)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    secs = n / SR
    return secs / best, f"{windows} windows ({secs:.1f} s of 16 kHz noise): log-mel + model (batch {windows}) + notes, torch fp32 CPU, {best:.2f} s wall"


def workload_config(args, world):
    if args.config == 3:
        return {"workload": CONFIG_TEXT[3], "songs": 1, "windows": 30, "window_batch": args.window_batch,
                "sharding": "one song" if world == 1 else f"the song's 30 windows split over {world} ranks, one final gather of the rolls",
                "cache": "L2 flushed between timed steps (a 512 MB buffer is rewritten); a step streams ~30 GB of activations"}
    per = TOTAL_SONGS // world
    return {"workload": CONFIG_TEXT[4], "songs_total": TOTAL_SONGS, "songs_per_gpu": per, "windows_per_song": 30,
            "window_batch": args.window_batch,
            "cache": "inputs larger than L2 (15.4 MB wave + ~1 GB of activations per window batch vs 126 MB L2)",
            "sharding": "songs over ranks, no hot-path collective; one final gather of the note records to rank 0 in the e2e leg"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, as restated by the oracle port (the reference
    itself is pure Python and not on the GPU box), on all host threads; each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    windows = 2
    vals = []
    for i in range(args.warmup + args.steps):
        v, desc = cpu_baseline_sample(threads, windows=windows)
        if i >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
            "warmup": args.warmup, "ms_per_step": 1e3 * windows * 8.192 / value, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, max(1, args.gpus)),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def frontend_10h(ex, steps=20, warmup=3, dump_dir=None):
    """BASELINE config 2: log-mel front-end over 150 four-minute songs (10 h, 576 M samples) resident in HBM; HBM roofline with
    the algorithmic bytes of SURVEY 8(d): 4 B per sample in + 4 B x 256 per frame out (intermediates never touch HBM)."""
    from etude_b200 import synth
    dev = ex.device
    n_songs = 150
    base = [torch.from_numpy(synth.noise(SONG_SAMPLES, 1234 + i)) for i in range(4)] + \
           [torch.from_numpy(synth.tones(SONG_SAMPLES, 4321 + i).astype(np.float32)) for i in range(2)]
    wave = torch.cat([base[i % len(base)] for i in range(n_songs)]).to(dev)      # both input classes of SURVEY 8(d)
    n_samples = [SONG_SAMPLES] * n_songs
    wave_off = (np.arange(n_songs, dtype=np.int64) * SONG_SAMPLES)
    frames = sum(1 + n // 256 for n in n_samples)
    alg_bytes = 4.0 * sum(n_samples) + 4.0 * 256 * frames
    feat = None
    for _ in range(warmup):
        feat = None
        feat, _ = ex.engine.logmel(wave, wave_off, n_samples)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        feat = None
        feat, _ = ex.engine.logmel(wave, wave_off, n_samples)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if dump_dir:
        dump_features(dump_dir, feat)
    del feat, wave
    torch.cuda.empty_cache()
    pk = peaks()
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    secs = sum(n_samples) / SR
    traffic = None   # DRAM bytes of one such launch, measured once with `ncu --set full` (same workload)
    tpath = os.path.join(ROOT, "profiles", "logmel_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        traffic = t["dram_bytes_read"] + t["dram_bytes_write"]
    return {"workload": CONFIG_TEXT[2] + " (150 x 4 min, noise + tones; 2.3 GB of samples in, 2.4 GB of features out, larger than L2)",
            "audio_s_per_s": secs / (ms * 1e-3), "ms_per_launch": ms, "launches": steps, "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"],
            "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk["source"] + ", HBM copy",
            "bytes_per_launch": alg_bytes, "bytes_per_audio_second": 128000}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=4, choices=(2, 3, 4))
    ap.add_argument("--songs", type=int, default=None, help="override the song count of config 4 (debugging only: not a BASELINE config)")
    ap.add_argument("--window-batch", type=int, default=None)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-windows", type=int, default=4)
    ap.add_argument("--frontend-microbench", action="store_true", help="same as --config 2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (seeded sample, under 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path; --impl reference has no device outputs")
    if args.frontend_microbench:
        args.config = 2
    if args.steps is None:
        args.steps = {4: 3, 3: 20, 2: 60}[args.config]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.window_batch is None:
        args.window_batch = 64 if args.config == 3 else 32
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from etude_b200 import AMTAPC_Extractor, ExtractorConfig, sharding
    from etude_b200.weights import default_state_dict
    sd = default_state_dict(seed=0)
    with tempfile.TemporaryDirectory() as tmp:     # the extractor reads the checkpoint in its constructor
        ckpt = os.path.join(tmp, "sd.pth")
        torch.save(sd, ckpt)
        ex = AMTAPC_Extractor(ExtractorConfig(), ckpt, device=dev, max_windows=args.window_batch)
    eng = ex.engine
    pk = peaks()

    if args.config == 2:
        if rank == 0:
            sampler = ClockSampler(local)
            sampler.start()
            fe = frontend_10h(ex, steps=args.steps, warmup=args.warmup, dump_dir=args.dump_outputs)
            clocks = sampler.stop()
            print(json.dumps({
                "metric": "logmel_frontend_audio_seconds_per_second", "value": fe["audio_s_per_s"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": fe["ms_per_launch"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": {"workload": fe["workload"], "cache": "inputs larger than L2"},
                "gpu_launches": args.steps, "clocks": clocks,
                "roofline": {"kernel": "logmel", "bound": "hbm", "achieved": fe["achieved"], "peak": fe["peak"], "unit": "GB/s", "frac": fe["frac"],
                             "traffic": fe["traffic"], "peak_source": fe["peak_source"], "bytes_per_launch": fe["bytes_per_launch"],
                             "avg_launch_ms": fe["ms_per_launch"]}}))
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- workload
    if args.config == 3:
        all_lengths = [SONG_SAMPLES]
        mine = [0]                                  # every rank holds the one song (window sharding splits its windows)
    else:
        total = args.songs if args.songs else TOTAL_SONGS
        all_lengths = [SONG_SAMPLES] * total
        mine = sharding.shard_songs(all_lengths, world)[rank]
    waves = [make_wave(i) for i in mine]
    n_samples = [len(w) for w in waves]
    wave_off = np.concatenate([[0], np.cumsum(n_samples)]).astype(np.int64)
    audio_seconds_total = sum(all_lengths) / SR    # the whole job, all ranks
    pinned = torch.empty(int(wave_off[-1]), dtype=torch.float32, pin_memory=True)
    pinned.numpy()[:] = np.concatenate(waves)
    wave_dev = pinned.to(dev)
    n_windows_mine = sum(sharding.windows_of(n) for n in n_samples)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev) if args.config == 3 else None

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    window_sharded = args.config == 3 and world > 1

    # ---------------- device-resident leg: waves in HBM -> log-mel -> model -> notes -> records on the host
    def step_device():
        if window_sharded:
            return sharding.extract_window_sharded(ex, wave_dev)
        return ex.extract_many(n_samples, as_dicts=False, wave_dev=wave_dev)

    def timed(step, steps):
        """K steps, CUDA events on the launching stream around every step (the L2 flush of config 3 sits between the
        steps, outside the events); returns the summed event time in ms."""
        evs = []
        for _ in range(steps):
            if flush is not None:
                flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = step()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs), out

    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    eng.profile_reset(timing=False)
    ms_total, recs = timed(step_device, args.steps)
    barrier()
    ms_total = max_over_ranks(ms_total)
    launches = eng.profile_read()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_notes(args.dump_outputs, [recs] if window_sharded else recs, mine)
    ms_per_step = ms_total / args.steps
    value = audio_seconds_total / (ms_per_step / 1e3)

    # ---------------- per-kernel-class timing: one extra, separately profiled pass (event pairs around every launch
    # serialise the streams a little, so it is kept out of the pass `value` is taken from)
    eng.profile_reset(timing=True)
    t_prof, _ = timed(step_device, 1)
    prof = eng.profile_read()
    eng.profile_reset(timing=False)

    # ---------------- end-to-end leg: pinned host waves -> note records on the host of rank 0, through the public API
    def step_e2e():
        if window_sharded:
            return sharding.extract_window_sharded(ex, waves[0])
        if dist is not None:
            got = ex.extract_many(waves, as_dicts=False, pinned=pinned)
            return sharding.gather_notes(got, mine, len(all_lengths), dst=0)      # = sharding.extract_sharded on a pre-sharded list
        return ex.extract_many(waves, as_dicts=False, pinned=pinned)

    step_e2e()
    barrier()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        if flush is not None:
            flush.fill_(1)
        recs_e2e = step_e2e()
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_value = audio_seconds_total / e2e_s
    d2h = int(sum(r.nbytes for r in recs_e2e)) if recs_e2e is not None else 0   # rank 0: every song's records
    h2d = int(4 * wave_off[-1])

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    model_classes = ("embed", "gemm_bias", "gemm_ln", "gemm_heads", "attention", "attention_fused", "chain")
    kernels = {}
    prof_ms = sum(p["ms"] for p in prof.values())
    for name, p in prof.items():
        if p["launches"] == 0:
            continue
        k = {"launches_per_step": p["launches"], "ms_per_step": p["ms"], "avg_launch_ms": p["ms"] / p["launches"],
             "share_of_kernel_time": p["ms"] / prof_ms if prof_ms > 0 else None}
        if p["flops"] > 0 and p["ms"] > 0:
            k["tflops"] = p["flops"] / (p["ms"] * 1e-3) / 1e12
        if p["bytes"] > 0 and p["ms"] > 0:
            k["gbs"] = p["bytes"] / (p["ms"] * 1e-3) / 1e9
        kernels[name] = k
    dom = max((n for n in kernels if n in model_classes), key=lambda n: kernels[n]["ms_per_step"])
    dom_p = prof[dom]
    achieved = dom_p["flops"] / (dom_p["ms"] * 1e-3) / 1e12
    traffic = None   # DRAM bytes per launch of the dominant kernel: measured once with `ncu --set full`
    tpath = os.path.join(ROOT, "profiles", "chain_traffic.json")
    if dom == "chain" and os.path.exists(tpath):
        t = json.load(open(tpath))
        traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["flop"] * (dom_p["flops"] / dom_p["launches"])
    long_step = ms_per_step > 500.0     # a kernel timed inside a seconds-long step runs power-capped: sustained peak
    peak = pk["bf16_sustained"] if long_step else pk["bf16_burst"]
    roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "frac_of_burst_peak": achieved / pk["bf16_burst"],
                "frac_of_sustained_peak": achieved / pk["bf16_sustained"], "traffic": traffic,
                "traffic_note": "ncu-measured DRAM bytes per FLOP of a chain3 launch (profiles/chain_traffic.json) x FLOP per launch here (algorithmic: 1 536 B/token)",
                "peak_source": pk["source"] + (", sustained bf16 (kernel timed inside a seconds-long step)" if long_step else ", burst bf16 (short step)"),
                "flop_per_launch": dom_p["flops"] / dom_p["launches"], "avg_launch_ms": dom_p["ms"] / dom_p["launches"]}
    flops_exec = sum(prof[n]["flops"] for n in model_classes if n in prof)
    model_ms = sum(prof[n]["ms"] for n in model_classes if n in prof)
    fe = prof["logmel"]
    frontend = {"kernel": "logmel", "bound": "hbm", "achieved": fe["bytes"] / (fe["ms"] * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": fe["bytes"] / (fe["ms"] * 1e-3) / 1e9 / pk["hbm_gbs"], "traffic": None,
                "bytes_per_launch": fe["bytes"] / fe["launches"], "avg_launch_ms": fe["ms"] / fe["launches"],
                "note": "inside the step, launches of a few songs each; the 10 h microbench (BASELINE config 2) is `frontend_10h`"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "api": ("sharding.extract_window_sharded(host wave)" if window_sharded else
                        "AMTAPC_Extractor.extract_many(host waves)" + (" + sharding.gather_notes (final gather to rank 0)" if world > 1 else ""))
                       + " -> note records on the host",
                "bytes_note": "per rank H2D of its waves; D2H = every note record reaching rank 0's host"},
        "gpu_launches": int(sum(p["launches"] for p in launches.values())),
        "clocks": clocks,
        "roofline": roofline,
        "model": {"tflops_executed": flops_exec / (model_ms * 1e-3) / 1e12, "gflop_per_window_executed": flops_exec / n_windows_mine / 1e9,
                  "gflop_per_window_reference": FLOP_PER_WINDOW_REF / 1e9,
                  "tensor_util_of_sustained_peak": flops_exec / (ms_per_step * 1e-3) / 1e12 / pk["bf16_sustained"],
                  "tensor_util_of_burst_peak": flops_exec / (ms_per_step * 1e-3) / 1e12 / pk["bf16_burst"],
                  "note": "executed FLOPs of rank 0's windows over the whole step time (front-end, note decoding and the D2H of the notes included), per GPU"},
        "frontend": frontend,
        "kernels": kernels,
        "profiled_pass_ms": t_prof,
    }
    if args.config == 4 and world == 1:
        del wave_dev
        torch.cuda.empty_cache()
        line["frontend_10h"] = frontend_10h(ex)
    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, desc = cpu_baseline_sample(threads, windows=args.cpu_windows)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
