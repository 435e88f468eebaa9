"""CPU checks of the native WAV header reader (etude_b200/audio.py) against scipy.io.wavfile."""
import struct
import wave

import numpy as np
import pytest
from scipy.io import wavfile

from etude_b200 import audio

GUID_TAIL = b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"


def _fmt(tag, ch, sr, bits, block_align=None, ext=None):
    ba = ch * bits // 8 if block_align is None else block_align
    body = struct.pack("<HHIIHH", tag, ch, sr, sr * ba, ba, bits)
    if ext is not None:   # (valid_bits, sub_tag)
        body += struct.pack("<HHI", 22, ext[0], 0) + struct.pack("<H", ext[1]) + GUID_TAIL
    return body


def _chunk(cid, body, size=None):
    out = cid + struct.pack("<I", len(body) if size is None else size) + body
    return out + (b"\x00" if len(body) & 1 else b"")


def _riff(chunks, magic=b"RIFF"):
    body = b"WAVE" + b"".join(chunks)
    return magic + struct.pack("<I", len(body)) + body


def _samples(fmt, n, ch, seed=0):
    rng = np.random.default_rng(seed)
    if fmt == "u8":
        return rng.integers(0, 256, (n, ch), dtype=np.uint8)
    if fmt == "s16":
        return rng.integers(-32768, 32768, (n, ch), dtype=np.int16)
    if fmt == "s32":
        return rng.integers(-2**31, 2**31, (n, ch), dtype=np.int64).astype(np.int32)
    if fmt == "f32":
        return rng.standard_normal((n, ch)).astype(np.float32)
    return rng.standard_normal((n, ch))   # f64


CODES = {"u8": audio.PCM_U8, "s16": audio.PCM_S16, "s24": audio.PCM_S24, "s32": audio.PCM_S32, "f32": audio.PCM_F32, "f64": audio.PCM_F64}


def _read_raw(info):
    buf = np.zeros(info.data_bytes, np.uint8)
    audio.read_wav_data(info, buf)
    return buf


@pytest.mark.parametrize("fmt", ["u8", "s16", "s32", "f32", "f64"])
@pytest.mark.parametrize("ch", [1, 2, 6])
def test_scipy_written_files(tmp_path, fmt, ch):
    x = _samples(fmt, 1001, ch)
    p = tmp_path / f"{fmt}_{ch}.wav"
    wavfile.write(p, 22050, x if ch > 1 else x[:, 0])
    info = audio.read_wav_info(p)
    sr, ref = wavfile.read(p)
    ref = ref.reshape(len(ref), -1)
    assert (info.format, info.channels, info.sample_rate, info.n_frames) == (CODES[fmt], ch, sr, ref.shape[0])
    assert np.array_equal(_read_raw(info).view(ref.dtype).reshape(-1, ch), ref)


@pytest.mark.parametrize("ch", [1, 2, 6])
def test_s24_written_with_wave_module(tmp_path, ch):
    v = np.random.default_rng(1).integers(-2**23, 2**23, (777, ch)).astype(np.int32)
    raw = v.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    p = tmp_path / "s24.wav"
    with wave.open(str(p), "wb") as w:
        w.setnchannels(ch)
        w.setsampwidth(3)
        w.setframerate(48000)
        w.writeframes(raw)
    info = audio.read_wav_info(p)
    sr, ref = wavfile.read(p)   # int32 << 8
    assert (info.format, info.channels, info.sample_rate, info.n_frames, info.bytes_per_sample) == (audio.PCM_S24, ch, 48000, 777, 3)
    b = _read_raw(info).reshape(-1, 3).astype(np.int32)
    got = (b[:, 0] << 8 | b[:, 1] << 16 | b[:, 2] << 24).reshape(-1, ch)
    assert np.array_equal(got, ref.reshape(-1, ch)) and np.array_equal(got >> 8, v)


@pytest.mark.parametrize("sub", [(1, 16, 16, "<i2"), (3, 32, 32, "<f4"), (1, 32, 24, "<i4")])
def test_extensible_odd_list_and_trailing_chunks(tmp_path, sub):
    tag, bits, valid, dt = sub
    x = (np.arange(60, dtype=np.float64).reshape(20, 3) * 1000 - 7).astype(dt)
    data = x.tobytes()
    chunks = [_chunk(b"fmt ", _fmt(0xFFFE, 3, 44100, bits, ext=(valid, tag))), _chunk(b"LIST", b"INFOabc"),
              _chunk(b"data", data), _chunk(b"JUNK", b"12345"), _chunk(b"bext", b"x" * 10)]
    p = tmp_path / "ext.wav"
    p.write_bytes(_riff(chunks))
    info = audio.read_wav_info(p)
    assert (info.channels, info.sample_rate, info.n_frames) == (3, 44100, 20)
    assert info.format == (audio.PCM_F32 if tag == 3 else audio.PCM_S16 if bits == 16 else audio.PCM_S32)
    assert np.array_equal(_read_raw(info).view(dt).reshape(20, 3), x)
    if tag == 1 and bits == 16:
        _, ref = wavfile.read(p)
        assert np.array_equal(ref, x)


@pytest.mark.parametrize("size", [0, 0xFFFFFFFF, 10**6])
def test_streaming_data_sizes(tmp_path, size):
    x = np.arange(-50, 51, dtype=np.int16).reshape(-1, 1)
    data = x.tobytes() + b"\x01"      # a partial trailing frame is dropped
    p = tmp_path / "stream.wav"
    p.write_bytes(_riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16)), b"data" + struct.pack("<I", size) + data]))
    info = audio.read_wav_info(p)
    assert info.n_frames == 101
    assert np.array_equal(_read_raw(info).view("<i2"), x[:, 0])


REJECT = {
    "rifx": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16)), _chunk(b"data", b"\0\0")], magic=b"RIFX"),
    "rf64": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16)), _chunk(b"data", b"\0\0")], magic=b"RF64"),
    "bw64": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16)), _chunk(b"data", b"\0\0")], magic=b"BW64"),
    "adpcm": lambda: _riff([_chunk(b"fmt ", _fmt(2, 1, 8000, 4, block_align=256)), _chunk(b"data", b"\0" * 256)]),
    "alaw": lambda: _riff([_chunk(b"fmt ", _fmt(6, 1, 8000, 8)), _chunk(b"data", b"\0\0")]),
    "mulaw": lambda: _riff([_chunk(b"fmt ", _fmt(7, 1, 8000, 8)), _chunk(b"data", b"\0\0")]),
    "mpeg": lambda: _riff([_chunk(b"fmt ", _fmt(0x55, 2, 44100, 0, block_align=1)), _chunk(b"data", b"\0\0")]),
    "bits12": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 12, block_align=2)), _chunk(b"data", b"\0\0")]),
    "float16": lambda: _riff([_chunk(b"fmt ", _fmt(3, 1, 8000, 16)), _chunk(b"data", b"\0\0")]),
    "ext_unknown_guid": lambda: _riff([_chunk(b"fmt ", _fmt(0xFFFE, 1, 8000, 16, ext=(16, 2))), _chunk(b"data", b"\0\0")]),
    "zero_channels": lambda: _riff([_chunk(b"fmt ", _fmt(1, 0, 8000, 16, block_align=0)), _chunk(b"data", b"\0\0")]),
    "65_channels": lambda: _riff([_chunk(b"fmt ", _fmt(1, 65, 8000, 16)), _chunk(b"data", b"\0" * 130)]),
    "block_align": lambda: _riff([_chunk(b"fmt ", _fmt(1, 2, 8000, 16, block_align=2)), _chunk(b"data", b"\0\0")]),
    "no_fmt": lambda: _riff([_chunk(b"data", b"\0\0")]),
    "no_data": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16))]),
    "truncated_riff": lambda: b"RIFF\x10\x00",
    "truncated_fmt": lambda: _riff([_chunk(b"fmt ", _fmt(1, 1, 8000, 16))])[:30],
    "not_wave": lambda: b"RIFF" + struct.pack("<I", 4) + b"AVI ",
}


@pytest.mark.parametrize("case", sorted(REJECT))
def test_rejections_name_the_file(tmp_path, case):
    p = tmp_path / f"bad_{case}.wav"
    p.write_bytes(REJECT[case]())
    with pytest.raises(ValueError, match=f"bad_{case}.wav"):
        audio.read_wav_info(p)


def test_raw_layout_aligns_every_file(tmp_path):
    infos = []
    for i, n in enumerate([3, 8, 5]):
        p = tmp_path / f"{i}.wav"
        wavfile.write(p, 8000, np.zeros((n, 1), np.uint8))
        infos.append(audio.read_wav_info(p))
    offs, total = audio.raw_layout(infos)
    assert offs == [0, 8, 16] and total == 24
