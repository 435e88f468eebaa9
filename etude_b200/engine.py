"""Device engine: owns the C-ABI handle, its workspace and the device buffers of one GPU.

PyTorch is used only for plumbing (device memory, streams, pinned host buffers); all arithmetic of the hot path
runs in libetude_b200.so.  No method here has a PyTorch or CPU fallback.
"""
import ctypes

import numpy as np
import torch

from . import _lib

N_BIN, N_FRAME, MARGIN, N_NOTE, N_VEL = 256, 512, 32, 88, 128
WIN_ROWS = N_FRAME + 2 * MARGIN
MODE_VELOCITY = {"ignore_zero": 0, "org": 1}
MODE_OFFSET = {"shorter": 0, "longer": 1, "offset": 2}


def feature_rows(n_samples):
    """Rows of a song's padded feature block: 32 + T_pad + 32 (reference extractor.py:210-213)."""
    t = 1 + int(n_samples) // 256
    return (t + N_FRAME - 1) // N_FRAME * N_FRAME + 2 * MARGIN


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


NOTE_DTYPE = np.dtype([("pitch", np.int32), ("velocity", np.int32), ("onset", np.float64), ("offset", np.float64)])


def _take_notes(ptr, total):
    """Copies the `total` etude_note_t records at `ptr` (library-owned pinned memory, valid until the next etude_notes call)
    into a numpy structured array the caller owns (the plain etude_notes entry point; Engine.notes uses begin/fetch)."""
    if total <= 0:
        return np.zeros(0, dtype=NOTE_DTYPE)
    raw = (ctypes.c_uint8 * (total * NOTE_DTYPE.itemsize)).from_address(ctypes.cast(ptr, ctypes.c_void_p).value)
    return np.frombuffer(raw, dtype=NOTE_DTYPE).copy()


def _pinned_records(total):
    """A caller-owned structured array of `total` records over pinned host memory (torch's caching host allocator: recycled
    blocks, no cudaHostAlloc per call); the array keeps the allocation alive."""
    buf = torch.empty(max(1, total) * NOTE_DTYPE.itemsize, dtype=torch.uint8, pin_memory=True)
    return buf.numpy().view(NOTE_DTYPE)[:total]


class Engine:
    def __init__(self, weight_blob, device, max_windows=32):
        if not torch.cuda.is_available():
            raise _lib.EtudeError("etude_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.EtudeError(f"etude_b200 runs on CUDA devices only, got {self.device}")
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        self.lib = _lib.load()
        blob = np.ascontiguousarray(weight_blob, dtype=np.float32)
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_create(self.index, blob.ctypes.data, blob.size, ctypes.byref(self._h)), "etude_create")
        self.n_frame = int(self.lib.etude_n_frame(self._h))                 # 512 (AMT-APC extractor) or 128 (HFT_Transformer)
        self.win_rows = self.n_frame + 2 * MARGIN
        limit = int(self.lib.etude_max_windows(self._h))
        if int(max_windows) < 1:
            raise ValueError(f"max_windows must be >= 1, got {max_windows}")
        self.max_windows = min(int(max_windows), limit)                     # the library takes at most `limit` windows per call
        self._ws = None

    def close(self):
        if getattr(self, "_h", None):
            self.lib.etude_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _workspace(self, n_windows):
        need = self.lib.etude_workspace_bytes(self._h, int(n_windows))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    # ------------------------------------------------------------------ front-end
    def ingest(self, pcm, sr_in, sr_out=16000):
        """Channel mean + sinc resampling on the device (reference extractor.py:181-184).  pcm: float32 [C, N] or [N]
        (host or device); returns a 1-D device tensor of ceil(sr_out * N / sr_in) samples."""
        x = torch.as_tensor(pcm, dtype=torch.float32)
        if x.dim() == 1:
            x = x[None]
        x = x.to(self.device).contiguous()
        c, n = int(x.shape[0]), int(x.shape[1])
        n_out = int(self.lib.etude_resampled_length(n, int(sr_in), int(sr_out)))
        out = torch.empty(n_out, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_ingest(self._h, _ptr(x), c, n, int(sr_in), int(sr_out), _ptr(out), self._stream()), "etude_ingest")
        return out

    def ingest_reserve(self, sample_rates, sr_out=16000):
        """Builds the resampling tables of these input rates now (a synchronous upload each), not inside a pipeline."""
        rates = sorted({int(r) for r in sample_rates})
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_ingest_reserve(self._h, (ctypes.c_int * max(1, len(rates)))(*rates), len(rates), int(sr_out)),
                       "etude_ingest_reserve")

    def ingest_pcm(self, raw_dev, infos, sr_out=16000):
        """Raw PCM of many WAV files (audio.WavInfo) in one launch: ``raw_dev`` is a uint8 CUDA tensor holding their data
        chunks at audio.raw_layout(infos).  Returns (wave_dev, wave_off, n_samples): the songs' mono ``sr_out`` waves back
        to back in one fp32 tensor, as ``ingest`` returns them for the same samples converted to float."""
        from .audio import raw_layout
        offs, total = raw_layout(infos)
        if not (raw_dev.is_cuda and raw_dev.dtype == torch.uint8 and raw_dev.numel() >= total):
            raise ValueError(f"raw_dev must be a uint8 CUDA tensor of at least {total} bytes")
        n_samples = [int(self.lib.etude_resampled_length(i.n_frames, int(i.sample_rate), int(sr_out))) for i in infos]
        wave_off = np.concatenate([[0], np.cumsum(n_samples)]).astype(np.int64)
        songs = (_lib.PcmSong * len(infos))()
        for s, (info, o) in enumerate(zip(infos, offs)):
            songs[s] = _lib.PcmSong(o, info.n_frames, info.frame_bytes, info.bytes_per_sample, int(wave_off[s]), info.channels,
                                    info.sample_rate, info.format, 0)
        out = torch.empty(max(1, int(wave_off[-1])), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_ingest_pcm(self._h, _ptr(raw_dev), songs, len(infos), int(sr_out), _ptr(out), self._stream()),
                       "etude_ingest_pcm")
        return out, wave_off[:-1], n_samples

    def logmel(self, wave_dev, wave_off, n_samples):
        """wave_dev: 1-D fp32 CUDA tensor holding the songs back to back.  Returns (feat [rows,256], feat_row_off)."""
        rows = [feature_rows(n) for n in n_samples]
        row_off = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
        feat = torch.empty((int(row_off[-1]), N_BIN), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_logmel(self._h, _ptr(wave_dev), _lib.i64_array(wave_off), _lib.i64_array(n_samples),
                                             len(n_samples), _ptr(feat), _lib.i64_array(row_off[:-1]), self._stream()),
                       "etude_logmel")
        return feat, row_off

    def logmel_layout(self, wave_dev, wave_off, n_samples, rows, front_rows, pad_value, pad_reflect):
        """Log-mel into blocks of `rows[s]` rows: front_rows pad rows, the T frames, pad to the end (etude_logmel_layout)."""
        row_off = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
        feat = torch.empty((int(row_off[-1]), N_BIN), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_logmel_layout(self._h, _ptr(wave_dev), _lib.i64_array(wave_off), _lib.i64_array(n_samples),
                                                    len(n_samples), _ptr(feat), _lib.i64_array(row_off[:-1]), _lib.i64_array(rows),
                                                    int(front_rows), float(pad_value), int(bool(pad_reflect)), self._stream()),
                       "etude_logmel_layout")
        return feat, row_off

    # ------------------------------------------------------------------ model
    @staticmethod
    def _roll_ptrs(rolls):
        return (ctypes.c_void_p * 4)(*[t.data_ptr() for t in rolls]) if rolls is not None else None

    def forward_windows(self, feat, win_rows, out_rows, rolls_B, rolls_A=None, vel_logits_A=None, vel_logits_B=None,
                        attention=None, keep=None, enc_in=None):
        """Runs the model on len(out_rows) windows in chunks of ``max_windows``; writes the rolls in place.

        ``rolls_B=None`` skips the time-axis half (frequency-axis outputs only); ``keep=(first, count)`` writes only those
        frames of every window, at rows out_rows[w] .. + count (the overlapped windows of HFT_Transformer._transcript_stride);
        ``enc_in`` (fp32 [n * n_frame * 256, 256]) starts from a given encoder output instead of the features (decode)."""
        n = len(out_rows)
        F = self.n_frame
        ws = self._workspace(min(n, self.max_windows))
        arr_b, arr_a = self._roll_ptrs(rolls_B), self._roll_ptrs(rolls_A)
        with torch.cuda.device(self.index):
            for s in range(0, n, self.max_windows):
                e = min(n, s + self.max_windows)
                k = e - s

                def sl(t, per):
                    return ctypes.c_void_p(t.data_ptr() + s * per * t.element_size()) if t is not None else None

                if enc_in is not None:
                    _lib.check(self.lib.etude_decode_windows(
                        self._h, sl(enc_in, F * N_BIN * 256), _lib.i64_array(out_rows[s:e]), k, arr_a, arr_b,
                        sl(vel_logits_A, F * N_NOTE * N_VEL), sl(vel_logits_B, F * N_NOTE * N_VEL),
                        sl(attention, F * 4 * N_NOTE * N_BIN), _ptr(ws), ws.numel(), self._stream()), "etude_decode_windows")
                elif keep is not None:
                    _lib.check(self.lib.etude_forward_windows_stride(
                        self._h, _ptr(feat), _lib.i64_array(win_rows[s:e]), _lib.i64_array(out_rows[s:e]), k, arr_a, arr_b,
                        int(keep[0]), int(keep[1]), _ptr(ws), ws.numel(), self._stream()), "etude_forward_windows_stride")
                else:
                    _lib.check(self.lib.etude_forward_windows(
                        self._h, _ptr(feat), _lib.i64_array(win_rows[s:e]), _lib.i64_array(out_rows[s:e]), k, arr_a, arr_b,
                        sl(vel_logits_A, F * N_NOTE * N_VEL), sl(vel_logits_B, F * N_NOTE * N_VEL),
                        sl(attention, F * 4 * N_NOTE * N_BIN), _ptr(ws), ws.numel(), self._stream()),
                        "etude_forward_windows")

    def encode_windows(self, feat, win_rows):
        """Encoder half only: fp32 [n, n_frame, 256, 256] (= Encoder_SPEC2MIDI.forward's output, amt_apc.py:120)."""
        n = len(win_rows)
        F = self.n_frame
        out = torch.empty((n, F, N_BIN, 256), dtype=torch.float32, device=self.device)
        ws = self._workspace(min(n, self.max_windows))
        with torch.cuda.device(self.index):
            for s in range(0, n, self.max_windows):
                e = min(n, s + self.max_windows)
                _lib.check(self.lib.etude_encode_windows(self._h, _ptr(feat), _lib.i64_array(win_rows[s:e]), e - s, _ptr(out[s]), _ptr(ws),
                                                         ws.numel(), self._stream()), "etude_encode_windows")
        return out

    @staticmethod
    def alloc_rolls(rows, device):
        return [torch.zeros((rows, N_NOTE), dtype=torch.float32, device=device) for _ in range(3)] + \
               [torch.zeros((rows, N_NOTE), dtype=torch.int8, device=device)]

    # ------------------------------------------------------------------ notes
    def notes_reserve(self, max_rows, max_songs):
        """Sizes the note stage's device scratch once (the largest notes batch), so no later call has to grow it."""
        with torch.cuda.device(self.index):
            _lib.check(self.lib.etude_notes_reserve(self._h, int(max_rows), int(max_songs)), "etude_notes_reserve")

    def notes(self, onset, offset, mpe, velocity, song_row_off, song_rows, thred_onset, thred_offset, thred_mpe,
              mode_velocity="ignore_zero", mode_offset="shorter", note_min=21, hop_sec=256 / 16000):
        n_songs = len(song_rows)
        counts = (ctypes.c_int64 * n_songs)()
        with torch.cuda.device(self.index):
            # first half of the round trip: every kernel + the per-song counts; second half: the records, straight into the
            # pinned array that is returned (no staging copy on the host)
            _lib.check(self.lib.etude_notes_begin(
                self._h, _ptr(onset), _ptr(offset), _ptr(mpe), _ptr(velocity), _lib.i64_array(song_row_off),
                _lib.i64_array(song_rows), n_songs, int(note_min), float(hop_sec), float(thred_onset), float(thred_offset),
                float(thred_mpe), MODE_VELOCITY.get(mode_velocity, 1), MODE_OFFSET.get(mode_offset, 0), counts, self._stream()),
                "etude_notes_begin")
            total = int(sum(counts))
            rec = _pinned_records(total)
            if total > 0:
                _lib.check(self.lib.etude_notes_fetch(self._h, ctypes.c_void_p(rec.ctypes.data), total, self._stream()), "etude_notes_fetch")
        res, pos = [], 0
        for s in range(n_songs):
            res.append(rec[pos : pos + counts[s]])
            pos += counts[s]
        return res


def _profile_methods():
    def profile_reset(self, timing=False):
        _lib.check(self.lib.etude_profile_reset(self._h, int(bool(timing))), "etude_profile_reset")

    def profile_read(self):
        """{class: {"ms", "launches", "flops", "bytes"}} since the last reset (synchronises the device)."""
        n = self.lib.etude_profile_classes()
        ms, fl, by = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
        la = (ctypes.c_int64 * n)()
        _lib.check(self.lib.etude_profile_read(self._h, ms, la, fl, by), "etude_profile_read")
        return {self.lib.etude_profile_class_name(i).decode(): {"ms": ms[i], "launches": int(la[i]), "flops": fl[i], "bytes": by[i]}
                for i in range(n)}

    def profile_timeline(self, cap=65536):
        """[(class, start_ms, dur_ms)] of the launches of the last timed pass, in recording order."""
        st, du, cl = (ctypes.c_double * cap)(), (ctypes.c_double * cap)(), (ctypes.c_int32 * cap)()
        n = self.lib.etude_profile_timeline(self._h, st, du, cl, cap)
        if n < 0:
            _lib.check(n, "etude_profile_timeline")
        return [(self.lib.etude_profile_class_name(cl[i]).decode(), st[i], du[i]) for i in range(n)]

    Engine.profile_reset = profile_reset
    Engine.profile_read = profile_read
    Engine.profile_timeline = profile_timeline


_profile_methods()


def notes_to_dicts(rec):
    """Structured note array -> the reference's list of dicts (extractor.py:406)."""
    return [{"pitch": int(p), "onset": float(a), "offset": float(b), "velocity": int(v)}
            for p, a, b, v in zip(rec["pitch"].tolist(), rec["onset"].tolist(), rec["offset"].tolist(), rec["velocity"].tolist())]
