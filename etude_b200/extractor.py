"""Host-side mirror of ``etude/data/extractor.py``: same class, method names, arguments and outputs, with the
arithmetic done by the sm_100a kernels of libetude_b200.so.

    AMTAPC_Extractor(config, model_path, device="auto")            reference extractor.py:121-146
        .extract(audio_path, output_json_path, output_midi_path)   148-176
        ._wav2feature(audio_path) -> Tensor[T, 256]                178-197
        ._transcript(a_feature, ...) -> 8 ndarrays                 199-253
        ._mpe2note(a_onset, a_offset, a_mpe, a_velocity, ...)      256-418
        ._note2midi / ._note2json                                  421-446
    + extract_many(waves)   additive batch API (the reference is one song, batch 1)
    + extract_files(paths)  the same pipeline from WAV files (raw PCM converted and resampled on the device)

Differences from the reference, all deliberate: CUDA only (no cpu/mps path, no fallback); default ExtractorConfig
shapes only; windows are processed in batches and rolls stay on the device between the stages.
"""
import json
from pathlib import Path
from typing import Optional, Union

import numpy as np
import torch

from . import audio as _audio
from . import config as _config
from . import engine as _engine
from .model import Decoder_SPEC2MIDI as Decoder
from .model import Encoder_SPEC2MIDI as Encoder
from .model import _Spec2MIDI
from .weights import pack_state_dict

N_FRAME, MARGIN, N_BIN, N_NOTE = 512, 32, 256, 88


def _load_model(config, path_model, device, max_windows=32):
    """Reference: extractor.py:78-113.  ``strict=False``: absent keys keep their default initialisation."""
    _config.validate(config)
    encoder = Encoder(n_margin=config.input.margin_b, n_frame=config.input.num_frame, n_bin=config.feature.n_bins,
                      cnn_channel=config.model.cnn_channel, cnn_kernel=config.model.cnn_kernel,
                      hid_dim=config.model.transformer_hid_dim, n_layers=config.model.encoder_n_layer,
                      n_heads=config.model.encoder_n_head, pf_dim=config.model.transformer_pf_dim,
                      dropout=config.model.dropout, device=device)
    decoder = Decoder(n_frame=config.input.num_frame, n_bin=config.feature.n_bins, n_note=config.midi.num_note,
                      n_velocity=config.midi.num_velocity, hid_dim=config.model.transformer_hid_dim,
                      n_layers=config.model.decoder_n_layer, n_heads=config.model.decoder_n_head,
                      pf_dim=config.model.transformer_pf_dim, dropout=config.model.dropout, device=device)
    model = _Spec2MIDI(encoder, decoder, sv_dim=0, max_windows=max_windows)
    state_dict = torch.load(path_model, weights_only=True, map_location="cpu")
    model.load_state_dict(state_dict, strict=False)
    model.to(device)
    model.eval()
    return model


def _pipeline_groups(n_songs, group_songs):
    """Song ranges of the extract_many pipeline: groups of ``group_songs`` with a 1, 2, ... ramp at both ends, so that the
    exposed head (staging + H2D of the first group) and tail (note decoding + D2H of the last group) are one song's worth."""
    sizes, left = [], n_songs
    head, tail, k = [], [], 1
    while k < group_songs and left - sum(head) - sum(tail) > 2 * group_songs:
        head.append(k)
        tail.append(k)
        k *= 2
    left -= sum(head) + sum(tail)
    mid = [group_songs] * (left // group_songs) + ([left % group_songs] if left % group_songs else [])
    sizes = head + mid + tail[::-1]
    out, a = [], 0
    for n in sizes:
        out.append((a, a + n))
        a += n
    assert a == n_songs
    return out


class AMTAPC_Extractor:
    """A pipeline for converting audio into note lists (JSON/MIDI) -- B200-native drop-in for the reference class."""

    def __init__(self, config, model_path: Union[str, Path], device: Union[str, torch.device] = "auto", max_windows: int = 32):
        if device == "auto":
            if not torch.cuda.is_available():
                raise RuntimeError("etude_b200.AMTAPC_Extractor needs a CUDA (sm_100a) device; there is no CPU/MPS fallback")
            self.device = torch.device("cuda", torch.cuda.current_device())
        else:
            self.device = torch.device(device)
            if self.device.type != "cuda":
                raise RuntimeError(f"etude_b200.AMTAPC_Extractor runs on CUDA only, got device={device!r}")
            if self.device.index is None:
                self.device = torch.device("cuda", torch.cuda.current_device())
        self.config = _config.validate(config)
        self.model = _load_model(self.config, model_path, self.device, max_windows=max_windows)
        self.engine = self.model.engine(self.device)

    # ------------------------------------------------------------------ reference API
    def extract(self, audio_path: str, output_json_path: str, output_midi_path: Optional[str] = None):
        feature = self._wav2feature(audio_path, _on_device=True)
        _, _, _, _, onset, offset, frame, velocity = self._transcript(feature, _on_device=True, _skip_A=True)
        notes = self._mpe2note(onset, offset, frame, velocity, thred_onset=self.config.infer.onset_threshold,
                               thred_offset=self.config.infer.offset_threshold, thred_mpe=self.config.infer.frame_threshold)
        min_duration = self.config.infer.min_duration
        self._note2json(notes, output_json_path, min_duration)
        if output_midi_path:
            self._note2midi(notes, output_midi_path, min_duration)

    def _wav2feature(self, audio_path: str, _on_device: bool = False) -> torch.Tensor:
        """wav -> log-mel [T, 256].  File decoding stays on torchaudio (extractor.py:180), except for WAV files where
        torchaudio cannot decode (no TorchCodec): those are read natively (audio.load_resampled).  The channel mean and the
        Resample(sr, 16000) of extractor.py:181-184 run in the CUDA ingest kernel, the MelSpectrogram + log (186-197) in
        the fused CUDA front-end."""
        wave_mono = _audio.load_resampled(self.engine, audio_path, int(self.config.feature.sr))
        feat = self.wave_to_feature(wave_mono)
        return feat if _on_device else feat.cpu()

    def wave_to_feature(self, wave_mono) -> torch.Tensor:
        """Mono 16 kHz samples (tensor / ndarray, host or device) -> device log-mel [T, 256] (un-padded view)."""
        w = torch.as_tensor(wave_mono, dtype=torch.float32).reshape(-1).to(self.device).contiguous()
        n = int(w.numel())
        feat, _ = self.engine.logmel(w, [0], [n])
        t = 1 + n // 256
        return feat[MARGIN : MARGIN + t]

    def _transcript(self, a_feature, sv=None, silent=True, mode="combination", ablation_flag=False, _on_device=False,
                    _skip_A=False):
        """Reference: extractor.py:199-253.  Returns the 8 arrays with T_pad rows (the padded tail is not trimmed); with
        ``mode != "combination"`` only the four frequency-axis arrays (extractor.py:236, 250-253) -- the time-axis half of the
        decoder is then not run at all.  ``sv`` / ``ablation_flag`` are accepted for signature parity: the style-vector branch
        is compiled out (sv_dim = 0, extractor.py:107) and the ablation unpacking of extractor.py:232 selects the same arrays."""
        combination = mode == "combination"
        if not combination and _skip_A:
            raise ValueError("_skip_A needs mode='combination' (the frequency-axis arrays are the only output otherwise)")
        if _skip_A and not _on_device:
            raise ValueError("_skip_A returns device tensors only: pass _on_device=True")
        feat = torch.as_tensor(a_feature, dtype=torch.float32).to(self.device)
        t = feat.shape[0]
        if feat.dim() != 2 or feat.shape[1] != N_BIN:
            raise ValueError(f"a_feature must be [T, {N_BIN}], got {tuple(feat.shape)}")
        t_pad = (t + N_FRAME - 1) // N_FRAME * N_FRAME
        padded = torch.full((t_pad + 2 * MARGIN, N_BIN), float(self.config.input.min_value), dtype=torch.float32, device=self.device)
        padded[MARGIN : MARGIN + t] = feat
        starts = list(range(0, t, N_FRAME))
        rolls_b = self.engine.alloc_rolls(t_pad, self.device) if combination else None
        rolls_a = None if _skip_A else self.engine.alloc_rolls(t_pad, self.device)
        self.engine.forward_windows(padded, starts, starts, rolls_b, rolls_a)
        outs = (list(rolls_a) if rolls_a is not None else [None] * 4) + (list(rolls_b) if combination else [])
        if _on_device:
            return tuple(outs)
        return tuple(o.cpu().numpy() for o in outs)

    def _mpe2note(self, a_onset=None, a_offset=None, a_mpe=None, a_velocity=None, thred_onset=0.5, thred_offset=0.5,
                  thred_mpe=0.5, mode_velocity="ignore_zero", mode_offset="shorter"):
        """Reference: extractor.py:256-418 (bit-exact on identical rolls).  Accepts ndarrays or device tensors."""
        rec = self._mpe2note_rec(a_onset, a_offset, a_mpe, a_velocity, thred_onset, thred_offset, thred_mpe, mode_velocity,
                                 mode_offset)
        return _engine.notes_to_dicts(rec)

    def _mpe2note_rec(self, a_onset, a_offset, a_mpe, a_velocity, thred_onset, thred_offset, thred_mpe,
                      mode_velocity="ignore_zero", mode_offset="shorter"):
        on = torch.as_tensor(a_onset, dtype=torch.float32).to(self.device).contiguous()
        off = torch.as_tensor(a_offset, dtype=torch.float32).to(self.device).contiguous()
        mpe = torch.as_tensor(a_mpe, dtype=torch.float32).to(self.device).contiguous()
        vel = torch.as_tensor(a_velocity).to(torch.int8).to(self.device).contiguous()
        hop_sec = float(self.config.feature.hop_sample / self.config.feature.sr)
        return self.engine.notes(on, off, mpe, vel, [0], [on.shape[0]], thred_onset, thred_offset, thred_mpe, mode_velocity,
                                 mode_offset, note_min=self.config.midi.note_min, hop_sec=hop_sec)[0]

    def _note2midi(self, notes, path_output, min_length=0.0):
        """Reference: extractor.py:421-429."""
        import pretty_midi
        midi = pretty_midi.PrettyMIDI()
        instrument = pretty_midi.Instrument(program=0)
        for note in notes:
            if note["offset"] - note["onset"] < min_length:
                continue
            instrument.notes.append(pretty_midi.Note(velocity=note["velocity"], pitch=note["pitch"], start=note["onset"],
                                                     end=note["offset"]))
        midi.instruments.append(instrument)
        midi.write(path_output)

    def _note2json(self, notes, path_output, min_length=0.0):
        """Reference: extractor.py:432-446."""
        filtered = []
        for note in notes:
            if note["offset"] - note["onset"] < min_length:
                continue
            filtered.append({"onset": note["onset"], "offset": note["offset"], "pitch": note["pitch"], "velocity": note["velocity"]})
        with open(path_output, "w", encoding="utf-8") as f:
            json.dump(filtered, f, ensure_ascii=False, indent=2)

    # ------------------------------------------------------------------ additive batch API
    def extract_many(self, waves, as_dicts=True, return_rolls=False, pinned=None, group_songs=4, notes_batch=12, wave_dev=None):
        """Transcribes many mono 16 kHz songs: host waves -> H2D -> fused log-mel -> the model over all windows in
        batches -> device note decoding -> D2H of the notes.

        Songs go through the model in groups of ``group_songs`` (1, 2, ... ramp at both ends) on the launching stream while
        the copy stream stages + uploads the next group's waves, and notes are decoded on a third stream in batches of
        about ``notes_batch`` songs: the walk of one (song, pitch) is serial, so a notes call takes the same ~2 x 8 ms for
        one song as for fifty, and the model kernels do not make progress beside it (tests/coresidency_diag.py) -- few, large
        notes calls cost least; their D2H and host work overlap the next groups' model.  Results do not depend on the
        grouping (every window is independent; notes are decoded per song).

        ``waves``: list of 1-D float32 arrays.  Returns one note list per song (dicts like ``_mpe2note``, or
        structured arrays with ``as_dicts=False``), before the ``min_duration`` filter of ``_note2json``.
        ``return_rolls=True`` processes everything as one group and also returns the device rolls.
        ``wave_dev``: the same songs back to back in one 1-D float32 tensor already on this device (``waves`` then only
        gives the lengths: arrays or plain sample counts) -- no staging, no H2D; everything else is the same pipeline.
        """
        if len(waves) == 0:
            return ([], None, [], []) if return_rolls else []
        n_samples = [int(w) if np.isscalar(w) else int(np.asarray(w).shape[0]) for w in waves]
        wave_off = np.concatenate([[0], np.cumsum(n_samples)]).astype(np.int64)
        total = int(wave_off[-1])
        if wave_dev is not None:
            if not (wave_dev.is_cuda and wave_dev.dtype == torch.float32 and wave_dev.dim() == 1 and wave_dev.numel() >= total):
                raise ValueError("wave_dev must be a 1-D float32 CUDA tensor holding all songs back to back")
            hv = None
        else:
            if pinned is None or pinned.numel() < total:
                pinned = torch.empty(total, dtype=torch.float32, pin_memory=True)
            hv = pinned.numpy()

        def stage(a, b, copy_s, main):   # host staging + H2D of songs [a, b) on the copy stream
            lo, hi = int(wave_off[a]), int(wave_off[b])
            if wave_dev is not None:   # already resident: a view, ready as soon as the caller's stream is
                ev = torch.cuda.Event()
                ev.record(main)
                return wave_dev[lo:hi], ev
            for w, o, n in zip(waves[a:b], wave_off[a:b], n_samples[a:b]):
                hv[o : o + n] = np.asarray(w, dtype=np.float32).reshape(-1)
            with torch.cuda.stream(copy_s):
                dev = pinned[lo:hi].to(self.device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_s)
            return dev, ev

        return self._pipeline(n_samples, stage, as_dicts, return_rolls, group_songs, notes_batch)

    def extract_files(self, audio_paths, output_json_paths=None, as_dicts=True, group_songs=4, notes_batch=12):
        """The bulk form of ``extract(path, json)``: WAV files -> notes through the ``extract_many`` pipeline.

        Every header is parsed first (audio.read_wav_info), so a file that is not a supported WAV or is too short (16 kHz
        length <= 1024 samples) raises ValueError before any device work.  The staging step of a group reads its files'
        data chunks into pinned memory, uploads the raw bytes and converts + resamples them on the device
        (Engine.ingest_pcm), all on the copy stream while the model runs the previous group.  Pinned memory is two groups
        of raw bytes, each buffer reused only after its upload has completed.

        Returns what ``extract_many`` returns.  With ``output_json_paths`` every file's notes are also written exactly as
        ``extract`` writes them (``min_duration`` filter, indent 2)."""
        paths = [str(p) for p in audio_paths]
        if output_json_paths is not None and len(output_json_paths) != len(paths):
            raise ValueError(f"{len(paths)} audio files but {len(output_json_paths)} JSON paths")
        if not paths:
            return []
        sr_out = int(self.config.feature.sr)
        infos = [_audio.read_wav_info(p) for p in paths]
        n_samples = [int(self.engine.lib.etude_resampled_length(i.n_frames, i.sample_rate, sr_out)) for i in infos]
        for info, n in zip(infos, n_samples):
            if n <= 1024:
                raise ValueError(f"{info.path}: {info.n_frames} frames at {info.sample_rate} Hz are {n} samples at {sr_out} Hz; "
                                 "the log-mel needs more than 1024")
        self.engine.ingest_reserve([i.sample_rate for i in infos if i.sample_rate != sr_out], sr_out)
        groups = _pipeline_groups(len(paths), int(group_songs)) if group_songs and group_songs > 0 else [(0, len(paths))]
        cap = max(_audio.raw_layout(infos[a:b])[1] for a, b in groups)
        bufs = [torch.empty(max(1, cap), dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        buf_ev = [None, None]   # H2D of each pinned buffer's last group
        turn = [0]

        def stage(a, b, copy_s, main):
            k = turn[0] % 2
            turn[0] += 1
            if buf_ev[k] is not None:
                buf_ev[k].synchronize()
            offs, nbytes = _audio.raw_layout(infos[a:b])
            host = bufs[k].numpy()
            for info, o in zip(infos[a:b], offs):
                _audio.read_wav_data(info, host[o : o + info.data_bytes])
            with torch.cuda.stream(copy_s):
                raw = bufs[k][:nbytes].to(self.device, non_blocking=True)
                buf_ev[k] = torch.cuda.Event()
                buf_ev[k].record(copy_s)
                dev, _, _ = self.engine.ingest_pcm(raw, infos[a:b], sr_out)
                ev = torch.cuda.Event()
                ev.record(copy_s)
            return dev, ev

        recs = self._pipeline(n_samples, stage, False, False, group_songs, notes_batch)
        dicts = [_engine.notes_to_dicts(r) for r in recs] if as_dicts or output_json_paths is not None else None
        for notes, path in zip(dicts or [], output_json_paths or []):
            self._note2json(notes, path, self.config.infer.min_duration)
        return dicts if as_dicts else recs

    def _pipeline(self, n_samples, stage, as_dicts, return_rolls, group_songs, notes_batch):
        """The extract_many pipeline from the 16 kHz waves on; ``stage(a, b, copy_s, main)`` puts songs [a, b) back to back
        on the device and returns (tensor, event after which it is complete)."""
        cfg = self.config.infer
        hop_sec = float(self.config.feature.hop_sample / self.config.feature.sr)
        n_songs = len(n_samples)
        if return_rolls or group_songs is None or group_songs <= 0:
            groups = [(0, n_songs)]
        else:
            groups = _pipeline_groups(n_songs, int(group_songs))
        if notes_batch is None or notes_batch <= 0:
            notes_batch = n_songs
        wave_off = np.concatenate([[0], np.cumsum(n_samples)]).astype(np.int64)
        song_rows = [_engine.feature_rows(n) - 2 * MARGIN for n in n_samples]          # T_pad per song
        song_row_off = np.concatenate([[0], np.cumsum(song_rows)]).astype(np.int64)
        rolls = self.engine.alloc_rolls(int(song_row_off[-1]), self.device)            # one set of rolls for the whole call (caller's stream)
        # the note stage's scratch for the largest batch it will see: decode() is called with at most notes_batch + one group
        worst = min(n_songs, int(notes_batch) + int(max(b - a for a, b in groups)))
        self.engine.notes_reserve(int(sum(sorted(song_rows, reverse=True)[:worst])), worst)

        caller = torch.cuda.current_stream(self.device)
        if getattr(self, "_side_streams", None) is None:
            self._side_streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
        copy_s, notes_s, model_s = self._side_streams
        # The model must not run on the legacy default stream: work there does not overlap the notes stream at all (12
        # model launches: 3 ms alone, 50 ms beside a notes call on the default stream, 8 ms on a stream of their own --
        # tests/coresidency_diag.py), so a caller on the default stream gets a dedicated model stream.
        main = model_s if caller.cuda_stream == 0 else caller
        main.wait_stream(caller)
        copy_s.wait_stream(main)
        notes_s.wait_stream(main)

        def decode(a, b, ev):  # note decoding + D2H of songs [a, b) on the notes stream, once their rolls are complete
            notes_s.wait_event(ev)
            with torch.cuda.stream(notes_s):
                return self.engine.notes(rolls[0], rolls[1], rolls[2], rolls[3], song_row_off[a:b].tolist(), song_rows[a:b],
                                         cfg.onset_threshold, cfg.offset_threshold, cfg.frame_threshold,
                                         note_min=self.config.midi.note_min, hop_sec=hop_sec)

        recs, keep = [], []
        decoded, ready, ev_ready = 0, 0, None     # songs [decoded, ready) have complete rolls once ev_ready fires
        staged = stage(*groups[0], copy_s, main)
        for gi, (a, b) in enumerate(groups):
            dev, ev_up = staged
            main.wait_event(ev_up)
            local_off = (wave_off[a:b] - wave_off[a]).astype(np.int64)
            with torch.cuda.stream(main):
                self.transcribe_device(dev, local_off, n_samples[a:b], rolls=rolls, row_base=int(song_row_off[a]))   # asynchronous
            ev_done = torch.cuda.Event()
            ev_done.record(main)
            keep.append(dev)                # device buffers stay alive until every stream is done with them
            if gi + 1 < len(groups):
                staged = stage(*groups[gi + 1], copy_s, main)
            if ready - decoded >= notes_batch:   # decode behind the model group just enqueued
                recs.extend(decode(decoded, ready, ev_ready))
                decoded = ready
            ready, ev_ready = b, ev_done
        recs.extend(decode(decoded, ready, ev_ready))
        main.wait_stream(notes_s)
        main.wait_stream(copy_s)
        caller.wait_stream(main)
        out = [_engine.notes_to_dicts(r) for r in recs] if as_dicts else recs
        if return_rolls:
            return out, rolls, song_row_off[:-1].tolist(), song_rows
        return out

    def transcribe_device(self, wave_dev, wave_off, n_samples, rolls=None, row_base=0):
        """Device-resident stages 1+2 for many songs: log-mel, then every window through the model.
        Returns (rolls_B [4 tensors of [sum T_pad, 88]], song_row_off, song_rows).  With ``rolls`` given the songs' rows are
        written from row ``row_base`` of those tensors (extract_many keeps one set of rolls for all its song groups)."""
        feat, feat_row_off = self.engine.logmel(wave_dev, wave_off, n_samples)
        song_rows = [_engine.feature_rows(n) - 2 * MARGIN for n in n_samples]  # T_pad per song
        song_row_off = int(row_base) + np.concatenate([[0], np.cumsum(song_rows)]).astype(np.int64)
        win_rows, out_rows = [], []
        for s, n in enumerate(n_samples):
            t = 1 + n // 256
            for i in range(0, t, N_FRAME):
                win_rows.append(int(feat_row_off[s]) + i)
                out_rows.append(int(song_row_off[s]) + i)
        if rolls is None:
            rolls = self.engine.alloc_rolls(int(song_row_off[-1]), self.device)
        self.engine.forward_windows(feat, win_rows, out_rows, rolls)
        return rolls, song_row_off[:-1].tolist(), song_rows
