"""WAV files read natively: RIFF/WAVE header parsing on the host, raw PCM to the device, conversion on the device.

    read_wav_info(path) -> WavInfo          the header only; nothing is decoded on the host
    read_wav_data(info, dst)                the data chunk straight into a caller's buffer (e.g. pinned memory)
    raw_layout(infos)                       byte offsets of many files back to back in one buffer (Engine.ingest_pcm)
    load_resampled(engine, path, sr_out)    torchaudio.load -> mean -> Resample, with the native reader for WAV files
                                            where torchaudio cannot decode (torchaudio >= 2.9 without TorchCodec)

Supported: WAVE_FORMAT_PCM u8 / s16 / s24 / s32, WAVE_FORMAT_IEEE_FLOAT f32 / f64 and WAVE_FORMAT_EXTENSIBLE with a PCM
or IEEE-float SubFormat (read at container width).  The samples become float32 on the device with FFmpeg's rules, the
values torchaudio.load returns where TorchCodec is installed (include/etude_b200.h, ETUDE_PCM_*).
"""
import os
import struct
from dataclasses import dataclass

import torch

PCM_U8, PCM_S16, PCM_S24, PCM_S32, PCM_F32, PCM_F64 = 1, 2, 3, 4, 5, 6
_PCM_BY_BITS = {8: PCM_U8, 16: PCM_S16, 24: PCM_S24, 32: PCM_S32}
_FLOAT_BY_BITS = {32: PCM_F32, 64: PCM_F64}
_TAG_PCM, _TAG_FLOAT, _TAG_EXTENSIBLE = 0x0001, 0x0003, 0xFFFE
_GUID_TAIL = b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"   # KSDATAFORMAT_SUBTYPE_* after the 2-byte tag
_COMPRESSED = {0x0002: "MS ADPCM", 0x0006: "A-law", 0x0007: "mu-law", 0x0011: "IMA ADPCM", 0x0050: "MPEG", 0x0055: "MPEG layer 3"}
MAX_CHANNELS = 64
RAW_ALIGN = 8   # raw_layout aligns every file to the largest sample size


@dataclass(frozen=True)
class WavInfo:
    path: str
    format: int            # PCM_* (ETUDE_PCM_*)
    channels: int
    sample_rate: int
    n_frames: int
    data_offset: int       # byte offset of the first sample in the file
    bytes_per_sample: int  # container width

    @property
    def frame_bytes(self):
        return self.channels * self.bytes_per_sample

    @property
    def data_bytes(self):
        return self.n_frames * self.frame_bytes


def _reject(path, why):
    raise ValueError(f"{path}: {why}")


def is_riff_wave(path):
    try:
        with open(path, "rb") as f:
            head = f.read(12)
    except OSError:
        return False
    return len(head) == 12 and head[:4] in (b"RIFF", b"RIFX", b"RF64", b"BW64") and head[8:12] == b"WAVE"


def _parse_fmt(path, body):
    if len(body) < 16:
        _reject(path, f"truncated fmt chunk ({len(body)} bytes)")
    tag, channels, rate, _, block_align, bits = struct.unpack_from("<HHIIHH", body)
    if tag == _TAG_EXTENSIBLE:
        if len(body) < 40:
            _reject(path, "truncated WAVE_FORMAT_EXTENSIBLE fmt chunk")
        valid_bits = struct.unpack_from("<H", body, 18)[0]
        sub = body[24:40]
        if sub[2:] != _GUID_TAIL:
            _reject(path, "WAVE_FORMAT_EXTENSIBLE with an unknown SubFormat GUID")
        tag = struct.unpack_from("<H", sub)[0]
        if valid_bits > bits:
            _reject(path, f"{valid_bits} valid bits in a {bits}-bit container")
    if tag == _TAG_PCM:
        fmt = _PCM_BY_BITS.get(bits)
    elif tag == _TAG_FLOAT:
        fmt = _FLOAT_BY_BITS.get(bits)
    else:
        name = _COMPRESSED.get(tag, "compressed or unknown")
        _reject(path, f"format tag 0x{tag:04x} ({name}) is not supported; only PCM and IEEE float WAV files are")
    if fmt is None:
        _reject(path, f"{bits}-bit {'PCM' if tag == _TAG_PCM else 'IEEE float'} samples are not supported")
    if channels < 1 or channels > MAX_CHANNELS:
        _reject(path, f"{channels} channels (1..{MAX_CHANNELS})")
    if rate < 1 or rate > 0x7FFFFFFF:
        _reject(path, f"sample rate {rate}")
    if block_align != channels * (bits // 8):
        _reject(path, f"block_align {block_align} != {channels} channels x {bits // 8} bytes")
    return fmt, channels, rate, bits // 8


def read_wav_info(path) -> WavInfo:
    """Parses the RIFF/WAVE header of ``path``.  Raises ValueError (naming the file and the reason) for anything the
    device ingest cannot read: big-endian RIFX, RF64/BW64, compressed formats, other bit depths, 0 or more than 64
    channels, an inconsistent block_align, a missing fmt/data chunk or a truncated header."""
    path = os.fspath(path)
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        head = f.read(12)
        if len(head) < 12:
            _reject(path, "truncated RIFF header")
        if head[:4] == b"RIFX":
            _reject(path, "big-endian RIFX files are not supported")
        if head[:4] in (b"RF64", b"BW64"):
            _reject(path, f"{head[:4].decode()} files are not supported")
        if head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            _reject(path, "not a RIFF/WAVE file")
        pos, fmt, data = 12, None, None
        while pos + 8 <= size:
            f.seek(pos)
            cid, csize = struct.unpack("<4sI", f.read(8))
            if cid == b"fmt ":
                if pos + 8 + csize > size:
                    _reject(path, "truncated fmt chunk")
                fmt = _parse_fmt(path, f.read(csize))
            elif cid == b"data":
                present = size - (pos + 8)
                # 0 / 0xFFFFFFFF / oversized: a header left by a streaming writer -- the bytes that are present
                n = present if csize in (0, 0xFFFFFFFF) or csize > present else csize
                data = (pos + 8, n)
                if n == present:
                    break
            pos += 8 + csize + (csize & 1)
    if fmt is None:
        _reject(path, "no fmt chunk")
    if data is None:
        _reject(path, "no data chunk")
    code, channels, rate, width = fmt
    return WavInfo(path, code, channels, rate, data[1] // (channels * width), data[0], width)


def read_wav_data(info: WavInfo, dst):
    """Reads the ``info.data_bytes`` bytes of the data chunk into ``dst`` (a writable buffer of at least that size, e.g.
    the numpy view of a pinned uint8 tensor), with no intermediate copy."""
    mv = memoryview(dst).cast("B")
    n = info.data_bytes
    if mv.nbytes < n:
        raise ValueError(f"{info.path}: destination holds {mv.nbytes} bytes, the data chunk {n}")
    with open(info.path, "rb") as f:
        f.seek(info.data_offset)
        got = 0
        while got < n:
            k = f.readinto(mv[got:n])
            if not k:
                _reject(info.path, f"data chunk ends after {got} of {n} bytes")
            got += k


def raw_layout(infos):
    """Byte offsets of the files' data chunks back to back (each aligned to RAW_ALIGN) and the total size."""
    offs, pos = [], 0
    for info in infos:
        offs.append(pos)
        pos += (info.data_bytes + RAW_ALIGN - 1) // RAW_ALIGN * RAW_ALIGN
    return offs, pos


def load_resampled(engine, audio_path, sr_out):
    """torchaudio.load(audio_path) -> channel mean -> Resample(sr, sr_out) on the device (reference extractor.py:180-184).
    Where torchaudio cannot load (ImportError: no TorchCodec) a RIFF/WAVE file goes through read_wav_info /
    Engine.ingest_pcm instead, with the same result as torchaudio.load returning the same float samples."""
    try:
        import torchaudio
        wave, sr = torchaudio.load(audio_path)
    except ImportError:
        if not is_riff_wave(audio_path):
            raise
        info = read_wav_info(audio_path)
        raw = torch.empty(max(1, raw_layout([info])[1]), dtype=torch.uint8, pin_memory=True)
        read_wav_data(info, raw.numpy())
        wave_dev, _, _ = engine.ingest_pcm(raw.to(engine.device, non_blocking=True), [info], sr_out)
        return wave_dev
    return engine.ingest(wave, int(sr), int(sr_out))
