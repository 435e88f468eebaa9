"""One-off A/B of etude_ingest between two builds of libetude_b200.so loaded side by side (e.g. the parent commit's
library against this tree's), on the seeded inputs of tests/test_kernels_gpu.py::test_ingest_vs_torchaudio and one
four-minute 44.1 kHz stereo song.  Records whether the outputs are bit-identical and each build's time per audio-second.

    python tools/ab_ingest_parent.py OLD_LIB.so [NEW_LIB.so] [--out FILE]

Prints one JSON line; --out also writes it to FILE.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from etude_b200 import _lib  # noqa: E402


def load(path):
    lib = ctypes.CDLL(path)
    for name in ("etude_create", "etude_destroy", "etude_ingest", "etude_resampled_length", "etude_last_error"):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SIGNATURES[name]
    blob = np.zeros(5614878, np.float32)
    h = ctypes.c_void_p()
    _lib.check(lib.etude_create(0, blob.ctypes.data, blob.size, ctypes.byref(h)), "etude_create", lib)
    return lib, h


def run(lib, h, x, sr):
    c, n = x.shape
    out = torch.empty(int(lib.etude_resampled_length(n, sr, 16000)), dtype=torch.float32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.etude_ingest(h, ctypes.c_void_p(x.data_ptr()), c, n, sr, 16000, ctypes.c_void_p(out.data_ptr()), st), "etude_ingest", lib)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old_lib")
    ap.add_argument("new_lib", nargs="?", default=_lib.LIB_PATH)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    old_path, new_path = args.old_lib, args.new_lib
    libs = {"old": load(old_path), "new": load(new_path)}
    cases = []
    for orig in (44100, 48000, 22050, 8000, 16000):        # test_ingest_vs_torchaudio's seeded inputs
        rng = np.random.default_rng(orig + 1)
        for channels, n in ((2, orig // 2 + 123), (1, 3 * orig + 5), (2, 7)):
            cases.append((f"{orig}Hz_{channels}ch_{n}", rng.uniform(-0.5, 0.5, (channels, n)).astype(np.float32), orig))
    rng = np.random.default_rng(7)
    song = rng.uniform(-0.5, 0.5, (2, 44100 * 240)).astype(np.float32)
    cases.append(("song_4min_44100Hz_2ch", song, 44100))
    identical = {}
    for name, x, sr in cases:
        xd = torch.from_numpy(x).cuda()
        a = run(*libs["old"], xd, sr).cpu().numpy()
        b = run(*libs["new"], xd, sr).cpu().numpy()
        identical[name] = bool(a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)))
    xd = torch.from_numpy(song).cuda()
    times = {"old": [], "new": []}
    for _ in range(5):          # alternate the builds
        for k in ("old", "new"):
            run(*libs[k], xd, 44100)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                run(*libs[k], xd, 44100)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / 5)
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = {"metric": "etude_ingest A/B (planar fp32 in, 16 kHz out)", "old_lib": os.path.basename(old_path),
           "bit_identical": identical, "all_identical": all(identical.values()),
           "song": "240 s, 44.1 kHz stereo", "ms_per_call": {k: float(np.median(v)) for k, v in times.items()},
           "us_per_audio_second": {k: float(np.median(v)) * 1e3 / 240 for k, v in times.items()},
           "speedup": float(np.median(times["old"]) / np.median(times["new"])), "gpu_power_limit": q}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    for lib, h in libs.values():
        lib.etude_destroy(h)


if __name__ == "__main__":
    main()
