"""GPU tests of native WAV ingest: Engine.ingest_pcm (raw PCM of many files -> 16 kHz mono in one launch) against
Engine.ingest on the same samples converted to float, AMTAPC_Extractor.extract_files against extract(), and the
_wav2feature fallback where torchaudio.load cannot decode."""
import ctypes
import json
import wave

import numpy as np
import pytest
import torch
from scipy.io import wavfile

from etude_b200 import _lib, audio, synth

pytestmark = pytest.mark.gpu

import gpu_diag as D  # noqa: E402

RATES = [8000, 11025, 16000, 22050, 32000, 44100, 48000, 96000]
FORMATS = ["u8", "s16", "s24", "s32", "f32", "f64"]


@pytest.fixture(scope="module")
def extractor():
    ex, _ = D.make_extractor(max_windows=4)
    return ex


def write_wav(path, fmt, sr, x):
    """x: float [n, ch] in [-1, 1] -> a file of that sample format; returns the float32 [ch, n] samples FFmpeg decodes."""
    n, ch = x.shape
    if fmt == "u8":
        v = np.clip(np.round(x * 127 + 128), 0, 255).astype(np.uint8)
        ref = (v.astype(np.float32) - 128) * np.float32(2.0 ** -7)
    elif fmt == "s16":
        v = np.clip(np.round(x * 32767), -32768, 32767).astype(np.int16)
        ref = v.astype(np.float32) * np.float32(2.0 ** -15)
    elif fmt == "s24":
        v = np.clip(np.round(x * 8388607), -8388608, 8388607).astype(np.int32)
        with wave.open(str(path), "wb") as w:
            w.setnchannels(ch)
            w.setsampwidth(3)
            w.setframerate(sr)
            w.writeframes(v.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes())
        _, dec = wavfile.read(path)   # int32 << 8
        ref = (dec.reshape(n, ch) >> 8).astype(np.float32) * np.float32(2.0 ** -23)
        return np.ascontiguousarray(ref.T)
    elif fmt == "s32":
        v = np.clip(np.round(x * 2147483647.0), -2**31, 2**31 - 1).astype(np.int32)
        ref = v.astype(np.float32) * np.float32(2.0 ** -31)
    elif fmt == "f32":
        v = x.astype(np.float32)
        ref = v
    else:
        v = x.astype(np.float64) * (1 + 1e-9)
        ref = v.astype(np.float32)
    wavfile.write(path, sr, v)
    return np.ascontiguousarray(ref.T)


def signal(n, ch, seed):
    rng = np.random.default_rng(seed)
    return np.clip(rng.uniform(-0.9, 0.9, (n, ch)) * rng.uniform(0.1, 1, (1, ch)), -1, 1)


def upload(infos, dev="cuda"):
    offs, total = audio.raw_layout(infos)
    host = np.zeros(max(1, total), np.uint8)
    for info, o in zip(infos, offs):
        audio.read_wav_data(info, host[o : o + info.data_bytes])
    return torch.from_numpy(host).to(dev)


@pytest.mark.parametrize("fmt", FORMATS)
def test_formats_and_rates_match_ingest(extractor, tmp_path, fmt):
    """ingest_pcm == Engine.ingest on the decoded float samples (bit for bit) and within 1e-5 of torchaudio's Resample."""
    import torchaudio
    eng = extractor.engine
    worst = 0.0
    for ch in (1, 2, 3):
        for sr in RATES:
            x = signal(sr // 3 + 37, ch, sr + ch)
            p = tmp_path / f"{fmt}_{ch}_{sr}.wav"
            ref_f = write_wav(p, fmt, sr, x)
            info = audio.read_wav_info(p)
            got, off, n = eng.ingest_pcm(upload([info]), [info], 16000)
            got = got[: n[0]].cpu().numpy()
            want = eng.ingest(ref_f, sr, 16000).cpu().numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (fmt, ch, sr)
            ta = torchaudio.transforms.Resample(sr, 16000)(torch.mean(torch.from_numpy(ref_f), dim=0)).numpy()
            worst = max(worst, float(np.abs(got - ta).max()))
    assert worst <= 1e-5, worst


def _lengths():
    # tile sizes of ingest_pcm_kernel: 5120 outputs at 44.1 kHz (32 super-periods x 160), 4096 at 48 kHz, 1024 at 16 kHz
    out = [(44100, 7), (44100, 20), (48000, 30), (8000, 3), (16000, 1), (22050, 11)]
    for sr, tile in ((44100, 5120), (48000, 4096), (16000, 1024)):
        g = np.gcd(sr, 16000)
        for n_out in (tile - 1, tile, tile + 1, 2 * tile + 1):
            n = n_out * (sr // g) // (16000 // g)
            while -(-(16000 // g) * n // (sr // g)) < n_out:
                n += 1
            out.append((sr, n))
    return out


def test_batched_call_equals_per_song_calls_and_keeps_guards(extractor, tmp_path):
    """Mixed formats, rates, channel counts and lengths (7-frame clips, clips shorter than the tap span, outputs at tile
    boundaries +-1, more songs than one launch holds) in one call: the same bits as one call per song, and sentinel-filled
    gaps between the destinations stay untouched."""
    eng = extractor.engine
    infos = []
    for i, (sr, n) in enumerate(_lengths() * 2):
        p = tmp_path / f"b{i}.wav"
        write_wav(p, FORMATS[i % 6], sr, signal(n, 1 + i % 3, i))
        infos.append(audio.read_wav_info(p))
    assert len(infos) > 24
    raw = upload(infos)
    n_out = [int(eng.lib.etude_resampled_length(i.n_frames, i.sample_rate, 16000)) for i in infos]
    guard = 13
    dst = np.concatenate([[guard], np.cumsum(np.array(n_out) + guard) + guard])[:-1].astype(np.int64)
    out = torch.full((int(dst[-1] + n_out[-1] + guard),), -7.25, dtype=torch.float32, device="cuda")
    offs, _ = audio.raw_layout(infos)
    songs = (_lib.PcmSong * len(infos))()
    for s, (info, o) in enumerate(zip(infos, offs)):
        songs[s] = _lib.PcmSong(o, info.n_frames, info.frame_bytes, info.bytes_per_sample, int(dst[s]), info.channels,
                                info.sample_rate, info.format, 0)
    _lib.check(eng.lib.etude_ingest_pcm(eng._h, ctypes.c_void_p(raw.data_ptr()), songs, len(infos), 16000,
                                        ctypes.c_void_p(out.data_ptr()), eng._stream()), "etude_ingest_pcm")
    got = out.cpu().numpy()
    mask = np.ones(got.shape, bool)
    for s, info in enumerate(infos):
        one, _, n = eng.ingest_pcm(upload([info]), [info], 16000)
        assert n[0] == n_out[s]
        assert np.array_equal(got[dst[s] : dst[s] + n_out[s]].view(np.uint32), one[: n[0]].cpu().numpy().view(np.uint32)), s
        mask[dst[s] : dst[s] + n_out[s]] = False
    assert np.all(got[mask] == -7.25)


def test_non_finite_samples_spread_like_ingest(extractor, tmp_path):
    eng = extractor.engine
    for sr in (44100, 48000, 16000):
        x = signal(sr, 2, 3).astype(np.float32)
        x[1000, 0] = np.inf
        x[5000, 1] = np.nan
        x[9000, :] = [-np.inf, np.inf]
        p = tmp_path / f"nf{sr}.wav"
        wavfile.write(p, sr, x)
        info = audio.read_wav_info(p)
        got, _, n = eng.ingest_pcm(upload([info]), [info], 16000)
        got = got[: n[0]].cpu().numpy()
        want = eng.ingest(np.ascontiguousarray(x.T), sr, 16000).cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got).any()
        assert np.array_equal(got[~np.isnan(got)], want[~np.isnan(want)])


def _four_files(tmp_path):
    specs = [("s16", 44100, 2), ("f32", 48000, 1), ("s24", 16000, 1), ("u8", 22050, 2)]
    paths, floats = [], {}
    for i, (fmt, sr, ch) in enumerate(specs):
        mono = synth.tones(int(sr * (2.5 + i)), 40 + i).astype(np.float64)
        x = np.stack([mono * (0.9 - 0.2 * c) for c in range(ch)], axis=1)
        p = tmp_path / f"song{i}_{fmt}.wav"
        floats[str(p)] = (write_wav(p, fmt, sr, x), sr)
        paths.append(str(p))
    return paths, floats


def test_extract_files_equals_extract(extractor, tmp_path, monkeypatch):
    import torchaudio
    paths, floats = _four_files(tmp_path)
    outs = [str(tmp_path / f"files{i}.json") for i in range(len(paths))]
    recs4 = extractor.extract_files(paths, outs, group_songs=4)
    recs1 = extractor.extract_files(paths, group_songs=1)
    assert recs1 == recs4
    monkeypatch.setattr(torchaudio, "load", lambda p: (torch.from_numpy(floats[str(p)][0]), floats[str(p)][1]))
    n_notes = 0
    for i, p in enumerate(paths):
        ref = str(tmp_path / f"extract{i}.json")
        extractor.extract(p, ref)
        assert open(outs[i], "rb").read() == open(ref, "rb").read(), p
        n_notes += len(json.load(open(ref)))
    assert n_notes > 0


def test_wav2feature_falls_back_to_native_reader(extractor, tmp_path, monkeypatch):
    import torchaudio

    from etude_b200 import hft
    from test_hft import _pickle_like_the_original, _seeded_hft_state_dict
    paths, floats = _four_files(tmp_path)
    pkl = tmp_path / "hft.pkl"
    _pickle_like_the_original(_seeded_hft_state_dict(), pkl)
    tr = hft.HFT_Transformer(hft.HFTConfig(), pkl, device="cuda:0")
    for model in (extractor, tr):
        monkeypatch.setattr(torchaudio, "load", lambda p: (torch.from_numpy(floats[str(p)][0]), floats[str(p)][1]))
        want = [model._wav2feature(p) for p in paths]

        def no_codec(p):
            raise ImportError("TorchCodec is required for load_with_torchcodec")
        monkeypatch.setattr(torchaudio, "load", no_codec)
        for p, w in zip(paths, want):
            got = model._wav2feature(p)
            assert got.shape == w.shape and torch.equal(got, w), p
        other = tmp_path / "song.flac"
        other.write_bytes(b"fLaC" + bytes(64))
        with pytest.raises(ImportError, match="TorchCodec"):
            model._wav2feature(str(other))


def test_bad_file_raises_before_any_launch(extractor, tmp_path):
    paths, _ = _four_files(tmp_path)
    bad = tmp_path / "alaw.wav"
    bad.write_bytes(open(paths[0], "rb").read(20) + b"\x06\x00" + open(paths[0], "rb").read()[22:])
    short = tmp_path / "short.wav"
    wavfile.write(short, 44100, np.zeros(2000, np.int16))
    eng = extractor.engine
    for extra in (bad, short):
        eng.profile_reset()
        with pytest.raises(ValueError, match=extra.name):
            extractor.extract_files(paths[:2] + [str(extra)] + paths[2:])
        assert sum(v["launches"] for v in eng.profile_read().values()) == 0


def test_profile_counts_ingest_launches(extractor, tmp_path):
    eng = extractor.engine
    infos = []
    for i in range(30):
        p = tmp_path / f"c{i}.wav"
        write_wav(p, "s16", 44100, signal(4410 + i, 2, i))
        infos.append(audio.read_wav_info(p))
    raw = upload(infos)
    eng.profile_reset()
    eng.ingest_pcm(raw, infos, 16000)
    prof = eng.profile_read()["ingest"]
    assert prof["launches"] == 2   # 24 songs per launch
    assert prof["bytes"] == sum(i.data_bytes for i in infos) + 4 * sum(-(-160 * i.n_frames // 441) for i in infos)
    assert prof["flops"] > 0
