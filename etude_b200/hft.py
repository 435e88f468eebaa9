"""Host-side mirror of ``etude/models/hft_transformer.py``: the hFT-Transformer transcriber of dataset preparation
(prepare.py:98-101), same class, method names, arguments and outputs, on the same sm_100a kernels as the AMT-APC extractor.

    HFT_Transformer(config, model_path, device="auto")                      hft_transformer.py:36-73
        .transcribe(input_wav_path, output_json_path)                        75-117
        ._wav2feature(f_wav) -> Tensor[T, 256]                               119-138   (pad_mode="constant")
        ._transcript(a_feature, mode="combination") -> 8 ndarrays           140-280   (128-frame windows)
        ._transcript_stride(a_feature, n_offset, mode) -> 8 ndarrays        282-460   (windows advance by 64 frames, the centre
                                                                                       half of each is kept: stitched on the device)
        ._mpe2note(...)                                                      462-674   (same algorithm as the extractor's)

The model is the same architecture with ``num_frame = 128`` (HFTConfig.input, schema.py:175-181): only
``decoder.pos_embedding_time`` changes shape, and ``etude_create`` picks the window length from the weight count.
The checkpoint is a pickled module (hft_transformer.py:26-33, 52-53); ``load_pickled_state_dict`` unpickles it WITHOUT the
original class definitions: every class from the checkpoint's ``model*`` / ``etude.models.amt_apc`` modules becomes a bare
``nn.Module`` subclass that only carries its parameters, and the state_dict is read off that tree.
"""
import io
import json
import pickle
from dataclasses import dataclass, field
from pathlib import Path
from typing import Union

import numpy as np
import torch
import torch.nn as nn

from . import audio as _audio
from . import engine as _engine
from .config import ExtractorMidiConfig
from .weights import layout, pack_state_dict

MARGIN, N_BIN = 32, 256


@dataclass
class HFTFeatureConfig:          # schema.py:161-172
    sr: int = 16000
    hop_sample: int = 256
    mel_bins: int = 256
    n_bins: int = 256
    fft_bins: int = 2048
    window_length: int = 2048
    log_offset: float = 1e-8
    window: str = "hann"
    pad_mode: str = "constant"


@dataclass
class HFTInputConfig:            # schema.py:175-181
    margin_b: int = 32
    margin_f: int = 32
    num_frame: int = 128
    min_value: float = -80.0


@dataclass
class HFTInferConfig:            # schema.py:184-192
    mode: str = "combination"
    thred_mpe: float = 0.5
    thred_onset: float = 0.75
    thred_offset: float = 0.5
    n_stride: int = 32
    bpm: float = 120.0


@dataclass
class HFTConfig:                 # schema.py:195-201
    feature: HFTFeatureConfig = field(default_factory=HFTFeatureConfig)
    input: HFTInputConfig = field(default_factory=HFTInputConfig)
    midi: ExtractorMidiConfig = field(default_factory=ExtractorMidiConfig)
    infer: HFTInferConfig = field(default_factory=HFTInferConfig)


def validate(config):
    ref = HFTConfig()
    for section, names in (("feature", ["sr", "hop_sample", "mel_bins", "n_bins", "fft_bins", "window_length", "log_offset"]),
                           ("input", ["margin_b", "margin_f", "num_frame"]), ("midi", ["num_note", "num_velocity"])):
        for n in names:
            got, want = getattr(getattr(config, section), n), getattr(getattr(ref, section), n)
            if got != want:
                raise ValueError(f"etude_b200 is compiled for hft.{section}.{n} = {want!r}; got {got!r} (no fallback path)")
    if config.feature.pad_mode not in ("constant", "reflect"):
        raise ValueError(f"hft.feature.pad_mode must be 'constant' or 'reflect', got {config.feature.pad_mode!r}")
    return config


class _Bare(nn.Module):
    """Stand-in for a class of the checkpoint's own modules: holds parameters / sub-modules, never runs."""


class _CheckpointUnpickler(pickle.Unpickler):
    """hft_transformer.py:26-33 without the reference package: tensors go through torch.load, the checkpoint's own classes
    (module ``model*`` in the original hFT-Transformer pickles, ``etude.models.amt_apc`` when re-saved from Etude) become
    parameter containers."""

    _stubs = {}

    def find_class(self, module, name):
        if module == "torch.storage" and name == "_load_from_bytes":
            return lambda b: torch.load(io.BytesIO(b), map_location="cpu", weights_only=True)
        if module.startswith("model") or module.startswith("etude.models"):
            key = (module, name)
            if key not in self._stubs:
                self._stubs[key] = type(name, (_Bare,), {"__module__": __name__})
            return self._stubs[key]
        return super().find_class(module, name)


def load_pickled_state_dict(model_path):
    """Pickled Model_SPEC2MIDI -> state_dict with the extractor's key names (``encoder.*`` / ``decoder.*``)."""
    with open(model_path, "rb") as f:
        model = _CheckpointUnpickler(f).load()
    if not isinstance(model, nn.Module):
        raise TypeError(f"{model_path}: expected a pickled torch module, got {type(model).__name__}")
    out = {}
    for k, v in model.state_dict().items():
        for src, dst in (("encoder_spec2midi.", "encoder."), ("decoder_spec2midi.", "decoder."), ("encoder.", "encoder."), ("decoder.", "decoder.")):
            if k.startswith(src):
                out[dst + k[len(src):]] = v
                break
    want = dict(layout(128))
    missing = [k for k in want if k not in out]
    if missing:
        raise KeyError(f"{model_path}: checkpoint lacks {len(missing)} parameters of the hFT-Transformer, e.g. {missing[:3]}")
    return out


class HFT_Transformer:
    """A fully integrated transcriber based on the hFT-Transformer pipeline -- B200-native drop-in for the reference class."""

    def __init__(self, config, model_path: Union[str, Path], device: Union[str, torch.device] = "auto", max_windows: int = 128):
        if device == "auto":
            if not torch.cuda.is_available():
                raise RuntimeError("etude_b200.HFT_Transformer needs a CUDA (sm_100a) device; there is no CPU/MPS fallback")
            self.device = torch.device("cuda", torch.cuda.current_device())
        else:
            self.device = torch.device(device)
            if self.device.type != "cuda":
                raise RuntimeError(f"etude_b200.HFT_Transformer runs on CUDA only, got device={device!r}")
            if self.device.index is None:
                self.device = torch.device("cuda", torch.cuda.current_device())
        self.config = validate(config)
        sd = load_pickled_state_dict(model_path)
        blob, _ = pack_state_dict(sd, strict=True, n_frame=self.config.input.num_frame)
        self.engine = _engine.Engine(blob, self.device, max_windows=max_windows)
        assert self.engine.n_frame == self.config.input.num_frame

    # ------------------------------------------------------------------ reference API
    def transcribe(self, input_wav_path: Union[str, Path], output_json_path: Union[str, Path]):
        """Reference: hft_transformer.py:75-117."""
        feature = self._wav2feature(input_wav_path, _on_device=True)
        n_stride = self.config.infer.n_stride
        mode = self.config.infer.mode
        if n_stride > 0:
            predictions = self._transcript_stride(feature, n_stride, mode=mode, _on_device=True, _skip_unused=True)
        else:
            predictions = self._transcript(feature, mode=mode, _on_device=True, _skip_unused=True)
        if mode == "combination":
            onset, offset, mpe, velocity = predictions[4], predictions[5], predictions[6], predictions[7]
        else:
            onset, offset, mpe, velocity = predictions[0], predictions[1], predictions[2], predictions[3]
        notes = self._mpe2note(a_onset=onset, a_offset=offset, a_mpe=mpe, a_velocity=velocity, thred_onset=self.config.infer.thred_onset,
                               thred_offset=self.config.infer.thred_offset, thred_mpe=self.config.infer.thred_mpe)
        output_path = Path(output_json_path)
        output_path.parent.mkdir(parents=True, exist_ok=True)
        with open(output_path, "w", encoding="utf-8") as f:
            json.dump(notes, f, ensure_ascii=False, indent=4)

    def _wav2feature(self, f_wav, _on_device: bool = False) -> torch.Tensor:
        """Reference: hft_transformer.py:119-138.  wav -> log-mel [T, 256] with ``pad_mode`` from the config ("constant").
        WAV files torchaudio cannot decode (no TorchCodec) are read natively (audio.load_resampled)."""
        wave_mono = _audio.load_resampled(self.engine, f_wav, int(self.config.feature.sr))
        feat = self.wave_to_feature(wave_mono)
        return feat if _on_device else feat.cpu()

    def wave_to_feature(self, wave_mono) -> torch.Tensor:
        w = torch.as_tensor(wave_mono, dtype=torch.float32).reshape(-1).to(self.device).contiguous()
        n = int(w.numel())
        t = 1 + n // 256
        feat, _ = self.engine.logmel_layout(w, [0], [n], [t], 0, float(self.config.input.min_value), self.config.feature.pad_mode == "reflect")
        return feat

    def _padded(self, a_feature, front, rows):
        feat = torch.as_tensor(a_feature, dtype=torch.float32).to(self.device)
        if feat.dim() != 2 or feat.shape[1] != N_BIN:
            raise ValueError(f"a_feature must be [T, {N_BIN}], got {tuple(feat.shape)}")
        padded = torch.full((rows, N_BIN), float(self.config.input.min_value), dtype=torch.float32, device=self.device)
        padded[front : front + feat.shape[0]] = feat
        return padded

    def _run(self, padded, win_rows, out_rows, n_out, mode, keep, on_device, skip_unused):
        combination = mode == "combination"
        rolls_a = None if (combination and skip_unused) else self.engine.alloc_rolls(n_out, self.device)
        rolls_b = self.engine.alloc_rolls(n_out, self.device) if combination else None
        self.engine.forward_windows(padded, win_rows, out_rows, rolls_b, rolls_a, keep=keep)
        outs = (list(rolls_a) if rolls_a is not None else [None] * 4) + (list(rolls_b) if combination else [])
        if on_device:
            return tuple(outs)
        return tuple(o.cpu().numpy() for o in outs)

    def _transcript(self, a_feature, mode="combination", _on_device=False, _skip_unused=False):
        """Reference: hft_transformer.py:140-280 (non-overlapping 128-frame windows)."""
        f = self.config.input.num_frame
        t = int(torch.as_tensor(a_feature).shape[0])
        t_pad = (t + f - 1) // f * f
        padded = self._padded(a_feature, self.config.input.margin_b, t_pad + self.config.input.margin_b + self.config.input.margin_f)
        starts = list(range(0, t, f))
        return self._run(padded, starts, starts, t_pad, mode, (0, f), _on_device, _skip_unused)

    def _transcript_stride(self, a_feature, n_offset, mode="combination", _on_device=False, _skip_unused=False):
        """Reference: hft_transformer.py:282-460.  Windows start every num_frame / 2 frames; window frames
        [n_offset, n_offset + num_frame / 2) are kept -- written by the heads epilogue straight to their rows of the rolls."""
        f = self.config.input.num_frame
        half = f // 2
        mb, mf = self.config.input.margin_b, self.config.input.margin_f
        if not (0 <= int(n_offset) <= half):
            raise ValueError(f"n_offset must be in [0, {half}], got {n_offset}")
        t = int(torch.as_tensor(a_feature).shape[0])
        tmp_len = t + mb + mf + half
        len_s = (tmp_len + half - 1) // half * half - tmp_len
        rows = (mb + int(n_offset)) + t + (len_s + mf + (half - int(n_offset)))
        padded = self._padded(a_feature, mb + int(n_offset), rows)
        starts = list(range(0, t, half))
        return self._run(padded, starts, starts, t + len_s, mode, (int(n_offset), half), _on_device, _skip_unused)

    def _mpe2note(self, a_onset=None, a_offset=None, a_mpe=None, a_velocity=None, thred_onset=0.5, thred_offset=0.5, thred_mpe=0.5,
                  mode_velocity="ignore_zero", mode_offset="shorter"):
        """Reference: hft_transformer.py:462-674 (the extractor's algorithm; bit-exact on identical rolls)."""
        on = torch.as_tensor(a_onset, dtype=torch.float32).to(self.device).contiguous()
        off = torch.as_tensor(a_offset, dtype=torch.float32).to(self.device).contiguous()
        mpe = torch.as_tensor(a_mpe, dtype=torch.float32).to(self.device).contiguous()
        vel = torch.as_tensor(a_velocity).to(torch.int8).to(self.device).contiguous()
        hop_sec = float(self.config.feature.hop_sample / self.config.feature.sr)
        rec = self.engine.notes(on, off, mpe, vel, [0], [on.shape[0]], thred_onset, thred_offset, thred_mpe, mode_velocity, mode_offset,
                                note_min=self.config.midi.note_min, hop_sec=hop_sec)[0]
        return _engine.notes_to_dicts(rec)
